"""GPU tests of the fused predict + top-k path (K5: selection in the GEMM epilogue, no [B,V] score matrix) and of
the pipelined dense scores kernel, against the CPU oracle's reference chain and against the dense CUDA path."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _engine(V, H=100, C=50, B=128, seed=42, **kw):
    from aaerec_b200.engine import AAEEngine
    eng = AAEEngine(V, H, C, max_batch=B, **kw)
    eng.init_uniform(seed)
    # spread the logits (the stock init gives nearly flat scores): scale the decoder output layer
    eng.Wd3.mul_(8.0)
    eng.bd3.mul_(8.0)
    return eng


def _upload(eng, X):
    eng.upload_csr(X.indptr.astype(np.int32), X.indices.astype(np.int32))


def _oracle_logits(eng, X):
    sd = {k: torch.as_tensor(v) for k, v in eng.state_dict().items()}
    from oracle import aae_oracle as O
    return O.OracleAAE(sd, n_code=eng.C).logits(X.toarray())


@pytest.mark.parametrize("mode", ["v2", "v1"])
@pytest.mark.parametrize("V,B,k", [(40000, 70, 100), (150001, 200, 20), (70000, 130, 500), (300000, 1100, 100)])
def test_fused_topk_matches_oracle_and_dense_path(V, B, k, mode, monkeypatch):
    """mode v2: TMA-multicast single-pass TF32 filter + exact fp32 re-scoring of the survivors (aae_predict_topk2; a
    cluster of 1, 2 or 4 row-chunk CTAs for these batch sizes); mode v1: the 3xTF32 filter (aae_predict_topk)."""
    from aaerec_b200.synth import synth_sets
    from oracle import aae_oracle as O
    if mode == "v1":
        monkeypatch.setenv("AAE_B200_TOPK", "v1")
    eng = _engine(V, B=B)
    X = synth_sets(B, V, 20, seed=V % 89)
    _upload(eng, X)
    assert eng.impl_for_scores() == 1
    assert int(__import__("aaerec_b200")._native.load().aae_predict_topk_work_bytes(B, V, k)) > 0
    fi, fv = eng.topk(B, k)
    assert eng.topk_fallbacks == 0, "threshold estimate failed on benign scores"
    assert eng.topk_mode == mode
    di, dv = eng.topk(B, k, fused=False)
    fi, fv, di, dv = fi.cpu().numpy(), fv.cpu().numpy(), di.cpu().numpy(), dv.cpu().numpy()
    if mode == "v1":
        np.testing.assert_array_equal(fv, dv)          # same kernel arithmetic -> identical logits
        np.testing.assert_array_equal(fi, di)
    else:
        # exact fp32 FMA re-scoring vs the dense path's 3xTF32 logits: equal to fp32 rounding; the rankings may differ
        # only where two logits are within that rounding of each other
        np.testing.assert_allclose(fv, dv, rtol=3e-6, atol=3e-6)
        md = fi != di
        assert md.mean() < 0.01
        assert np.all(np.abs(fv[md] - dv[md]) <= 3e-6 * np.maximum(1.0, np.abs(dv[md])))
    # against the reference chain on the oracle's logits (sigmoid + min-max scaling are monotone): indices agree
    # except where fp32 logits are within rounding of each other
    Z = _oracle_logits(eng, X)
    ref = O.rank_topk(Z, X.toarray(), k)
    rows = np.arange(B)[:, None]
    mism = fi != ref
    assert mism.mean() < 0.02
    assert np.all(np.abs(Z[rows, fi][mism] - Z[rows, ref][mism]) <= 2e-5 * np.maximum(1.0, np.abs(Z[rows, ref][mism])))
    assert not X.toarray()[rows, fi].any(), "a known item was recommended"


def test_fused_topk_v2_margin_guards_exactness():
    """The v2 filter runs on single-pass TF32 logits: with an output layer scaled so that the TF32 error is far larger
    than the gaps between neighbouring scores, the ranking must still equal the exact dense ranking (margin + exact
    re-scoring), or the batch must be reported and redone -- never a silently wrong list."""
    from aaerec_b200.synth import synth_sets
    V, B, k = 60000, 64, 100
    eng = _engine(V, B=B)
    eng.Wd3.mul_(6.0)                    # |logits| up to ~50: TF32 absolute error ~5e-2
    X = synth_sets(B, V, 20, seed=4)
    _upload(eng, X)
    fi, fv = eng.topk(B, k)
    di, dv = eng.topk(B, k, fused=False)
    fi, fv, di, dv = fi.cpu().numpy(), fv.cpu().numpy(), di.cpu().numpy(), dv.cpu().numpy()
    np.testing.assert_allclose(fv, dv, rtol=3e-6, atol=3e-5)
    md = fi != di
    assert np.all(np.abs(fv[md] - dv[md]) <= 3e-6 * np.maximum(1.0, np.abs(dv[md])))


def test_fused_topk_degenerate_scores_fall_back_exactly():
    """All logits equal (zero output layer): the candidate filter finds nothing above the threshold, the status word
    reports it and the batch is re-ranked densely -- still k distinct unknown items per row."""
    from aaerec_b200.synth import synth_sets
    V, B, k = 40000, 40, 50
    eng = _engine(V)
    eng.Wd3.zero_()
    eng.bd3.zero_()
    X = synth_sets(B, V, 10, seed=3)
    _upload(eng, X)
    idx, val = eng.topk(B, k)
    assert eng.topk_fallbacks == 1
    idx = idx.cpu().numpy()
    Xd = X.toarray()
    for b in range(B):
        assert len(set(idx[b].tolist())) == k and not Xd[b, idx[b]].any()
    assert float(val.abs().max()) == 0.0


@pytest.mark.parametrize("V,B", [(1000, 5), (9999, 300), (70001, 129)])
def test_pipelined_scores_kernel_matches_oracle(V, B):
    """Dense predict (aae.py:840-870): sigmoid probabilities of the pipelined tcgen05 scores kernel vs the oracle and
    vs the fp32 CUDA-core kernel, incl. ragged last tile / last chunk and more than one chunk of 128 rows."""
    from aaerec_b200.synth import synth_sets
    from aaerec_b200._native import call, ptr
    eng = _engine(V, B=B)
    X = synth_sets(B, V, 15, seed=5)
    _upload(eng, X)
    out = torch.full((B, V), -7.0, device=eng.dev)
    eng.scores(B, out, apply_sigmoid=True)
    sd = {k: torch.as_tensor(v) for k, v in eng.state_dict().items()}
    from oracle import aae_oracle as O
    want = O.OracleAAE(sd, n_code=eng.C).predict(X.toarray())
    np.testing.assert_allclose(out.cpu().numpy(), want, rtol=2e-5, atol=1e-7)
    ref = torch.empty(B, V, device=eng.dev)
    call("aae_dec_out_scores", ptr(eng.h2), B, eng.H, ptr(eng.Wd3), ptr(eng.bd3), V, 0, ptr(ref), V, 0, eng._stream())
    tc = torch.empty(B, V, device=eng.dev)
    call("aae_dec_out_scores", ptr(eng.h2), B, eng.H, ptr(eng.Wd3), ptr(eng.bd3), V, 0, ptr(tc), V, 1, eng._stream())
    torch.cuda.synchronize()
    np.testing.assert_allclose(tc.cpu().numpy(), ref.cpu().numpy(), rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("mode", ["v2", "v1"])
def test_sharded_fused_topk_offsets(mode, monkeypatch):
    """v_begin / Vloc handling of the fused paths: two engines owning the halves of the vocabulary (as two ranks
    would), candidates merged with aae_topk_merge == the single-shard result."""
    from aaerec_b200.synth import synth_sets
    from aaerec_b200._native import call, ptr
    lib = __import__("aaerec_b200")._native.load()
    if mode == "v1":
        monkeypatch.setenv("AAE_B200_TOPK", "v1")
    V, B, k, H, C = 90000, 64, 100, 100, 50
    full = _engine(V)
    sd = full.state_dict()
    X = synth_sets(B, V, 20, seed=21)
    _upload(full, X)
    fi, fv = full.topk(B, k)
    assert full.topk_mode == mode
    cv, ci = [], []
    for r in range(2):
        # emulate rank r of 2 without a process group: shard the weights by hand, feed the full h2
        lo, hi = (0, V // 2) if r == 0 else (V // 2, V)
        Wd3 = sd["dec.lin3.weight"][lo:hi].contiguous().cuda()
        bd3 = sd["dec.lin3.bias"][lo:hi].contiguous().cuda()
        idx = torch.empty(B, k, dtype=torch.int32, device="cuda")
        val = torch.empty(B, k, dtype=torch.float32, device="cuda")
        n_bad = torch.zeros(1, dtype=torch.int32, device="cuda")
        if mode == "v1":
            need = int(lib.aae_predict_topk_work_bytes(B, hi - lo, k))
            assert need > 0
            work = torch.empty(need, dtype=torch.uint8, device="cuda")
            call("aae_predict_topk", ptr(full.h2), B, H, ptr(Wd3), ptr(bd3), hi - lo, lo, ptr(full.indptr),
                 ptr(full.indices), k, 1, ptr(work), need, ptr(idx), ptr(val), ptr(n_bad), None)
        else:
            need = int(lib.aae_predict_topk2_work_bytes(B, hi - lo, k, H))
            nwp = int(lib.aae_pad_weights_floats(hi - lo, H))
            assert need > 0 and nwp > 0
            work = torch.empty(need, dtype=torch.uint8, device="cuda")
            wp = torch.empty(nwp, dtype=torch.float32, device="cuda")
            call("aae_pad_weights", ptr(Wd3), ptr(bd3), hi - lo, H, ptr(wp), ptr(wp[nwp - 64:]), None)
            call("aae_predict_topk2", ptr(full.h2), B, H, ptr(Wd3), ptr(bd3), ptr(wp), ptr(wp[nwp - 64:]), hi - lo, lo,
                 ptr(full.indptr), ptr(full.indices), k, ptr(work), need, ptr(idx), ptr(val), ptr(n_bad), None)
        assert int(n_bad.item()) == 0
        cv.append(val)
        ci.append(idx)
    cv = torch.cat(cv, 1).contiguous()
    ci = torch.cat(ci, 1).contiguous()
    oi = torch.empty(B, k, dtype=torch.int32, device="cuda")
    ov = torch.empty(B, k, dtype=torch.float32, device="cuda")
    call("aae_topk_merge", ptr(cv), ptr(ci), B, cv.shape[1], k, ptr(oi), ptr(ov), None)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(oi.cpu().numpy(), fi.cpu().numpy())
    np.testing.assert_array_equal(ov.cpu().numpy(), fv.cpu().numpy())
