"""TEST INFRASTRUCTURE ONLY -- regenerate tests/golden/*.npz from the real reference.

Run in the authoring container (needs /root/reference):

    python oracle/make_golden.py

For each case it runs the UNMODIFIED reference ``aaerec.aae.AdversarialAutoEncoder.fit``
/ ``.predict`` and ``aaerec.evaluation.remove_non_missing`` / ``argtopk`` on seeded
inputs and stores inputs, initial weights, per-step losses, final weights, predictions
and rankings.  ``tests/test_oracle.py`` pins ``oracle/aae_oracle.py`` against these
files; the GPU parity tests compare the CUDA path with the same files.
"""
import io
import os
import sys
import contextlib

import numpy as np
import scipy.sparse as sp
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "aae-recommender_b200"))

from oracle.reference_loader import load_reference  # noqa: E402
from aaerec_b200.synth import synth_sets  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _state(model):
    out = {}
    for pre, mod in (("enc", model.enc), ("dec", model.dec), ("disc", getattr(model, "disc", None))):
        if mod is None:     # plain AutoEncoder: no discriminator
            continue
        for k, v in mod.state_dict().items():
            out[pre + "." + k] = v.detach().cpu().numpy().copy()
    return out


def run_case(ref, name, n, V, H, C, B, epochs, dropout, cond_dim=0, data_seed=0, mean_len=6,
             store_weights=True, store_init=True, k=10, adversarial=True, model_kwargs=None, dae=False):
    aae = ref.aae
    if dae:                     # aaerec/dae.py:144-314 (SURVEY 8(f)-3): the reference's DenoisingAutoEncoder
        import aaerec.dae
        cls = aaerec.dae.DenoisingAutoEncoder
        adversarial = False
    else:
        cls = aae.AdversarialAutoEncoder if adversarial else aae.AutoEncoder
    steps_per_fit = ("ae_step", "disc_step", "gen_step") if adversarial else ("ae_step",)
    X = synth_sets(n, V, mean_len, min_len=2, seed=data_seed)
    conditions = None
    cond_data = None
    cond = None
    if cond_dim:
        cond = (np.random.RandomState(data_seed + 1).randn(n, cond_dim) * 0.5).astype(np.float32)

        class MatrixCondition(ref.condition.ConcatenationBasedConditioning):
            """precomputed float rows, concatenated on the code (condition.py:300-316, 363-369)"""

            def __init__(self, dim):
                self._d = dim

            def encode(self, inputs):
                return torch.as_tensor(inputs, dtype=torch.float32)

            def size_increment(self):
                return self._d
        conditions = ref.condition.ConditionList([("title", MatrixCondition(cond_dim))])
        cond_data = [cond]

    losses = []
    orig = {k_: getattr(cls, k_) for k_ in steps_per_fit}

    def wrap(fn_name):
        fn = orig[fn_name]

        def inner(self, *a, **kw):
            val = fn(self, *a, **kw)
            losses.append(val)
            return val
        return inner
    for k_ in orig:
        setattr(cls, k_, wrap(k_))
    init = {}
    try:
        torch.manual_seed(42)     # aae.py:27 executes this at import; redo it per case
        np.random.seed(42)
        model = cls(n_hidden=H, n_code=C, batch_size=B, n_epochs=epochs, dropout=dropout, conditions=conditions,
                    verbose=False, **(model_kwargs or {}))
        # capture the initial weights: replay the same construction order under the same seed
        from oracle.aae_oracle import init_params
        init = {k_: v.numpy().copy() for k_, v in init_params(V, H, C, C + cond_dim, seed=42).items()}
        torch.manual_seed(42)
        with contextlib.redirect_stdout(io.StringIO()):
            model.fit(X, condition_data=cond_data)
        final = _state(model)
        with contextlib.redirect_stdout(io.StringIO()):
            pred = model.predict(X[:40], condition_data=[cond[:40]] if cond_dim else None)
    finally:
        for k_, fn in orig.items():
            setattr(cls, k_, fn)
    Xd = X[:40].toarray()
    masked = ref.evaluation.remove_non_missing(pred, Xd, copy=True)
    topk = ref.evaluation.argtopk(masked, k)[1]
    out = dict(
        n=n, V=V, H=H, C=C, B=B, epochs=epochs, dropout=np.asarray(dropout, dtype=np.float64),
        cond_dim=cond_dim, k=k, adversarial=int(adversarial), dae=int(dae),
        noise_factor=np.float64((model_kwargs or {}).get("noise_factor", 0.2)),
        normalize_inputs=int((model_kwargs or {}).get("normalize_inputs", True)),
        prior_scale=np.float64((model_kwargs or {}).get("prior_scale") or 0.0),
        gen_lr=np.float64((model_kwargs or {}).get("gen_lr", 0.001)),
        reg_lr=np.float64((model_kwargs or {}).get("reg_lr", 0.001)),
        indptr=X.indptr.astype(np.int32), indices=X.indices.astype(np.int32),
        losses=np.asarray(losses, dtype=np.float64).reshape(-1, len(steps_per_fit)),
        pred=pred.astype(np.float32), masked=masked.astype(np.float32), topk=topk.astype(np.int64),
    )
    if cond_dim:
        out["cond"] = cond
    if store_weights:
        if store_init:
            for k_, v in init.items():
                out["init/" + k_] = v
        for k_, v in final.items():
            out["final/" + k_] = v
    else:
        for k_, v in final.items():
            out["abssum/" + k_] = np.float64(np.abs(v.astype(np.float64)).sum())
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "steps", len(losses) // len(steps_per_fit), "first", out["losses"][0], "last", out["losses"][-1])
    return out


def _matrix_condition(ref, dim):
    class MatrixCondition(ref.condition.ConcatenationBasedConditioning):
        """precomputed float rows, concatenated on the code (condition.py:300-316, 363-369)"""

        def __init__(self, d):
            self._d = d

        def encode(self, inputs):
            return torch.as_tensor(inputs, dtype=torch.float32)

        def size_increment(self):
            return self._d
    return ref.condition.ConditionList([("title", MatrixCondition(dim))])


def run_vae_case(ref, name, n, V, H, C, B, epochs, cond_dim=0, data_seed=0, mean_len=6, k=10, lr=0.001):
    """aaerec/vae.py:47-266 (SURVEY 8(f)-3): the UNMODIFIED reference VAE -- construction, fit, predict.  Per-step losses
    are captured by wrapping ``loss_function``; predict is run after ``torch.manual_seed(123)`` so that its eval-mode
    reparametrisation draws (vae.py:252-256) can be replayed."""
    import aaerec.vae
    cls = aaerec.vae.VAE
    X = synth_sets(n, V, mean_len, min_len=2, seed=data_seed)
    cond = conditions = cond_data = None
    if cond_dim:
        cond = (np.random.RandomState(data_seed + 1).randn(n, cond_dim) * 0.5).astype(np.float32)
        conditions = _matrix_condition(ref, cond_dim)
        cond_data = [cond]
    losses = []
    orig = cls.loss_function

    def recording(self, *a, **kw):
        val = orig(self, *a, **kw)
        losses.append(float(val))
        return val
    cls.loss_function = recording
    try:
        torch.manual_seed(42)      # vae.py:30 executes this at import; redo it per case
        np.random.seed(42)
        model = cls(V, V, n_hidden=H, n_code=C, lr=lr, batch_size=B, n_epochs=epochs, conditions=conditions,
                    verbose=False, device=torch.device("cpu"))
        init = {k_: v.detach().cpu().numpy().copy() for k_, v in model.state_dict().items()}
        with contextlib.redirect_stdout(io.StringIO()):
            model.fit(X, condition_data=cond_data)
        n_fit = len(losses)
        final = {k_: v.detach().cpu().numpy().copy() for k_, v in model.state_dict().items()}
        torch.manual_seed(123)
        with contextlib.redirect_stdout(io.StringIO()):
            pred = model.predict(X[:40], condition_data=[cond[:40]] if cond_dim else None)
    finally:
        cls.loss_function = orig
    masked = ref.evaluation.remove_non_missing(pred, X[:40].toarray(), copy=True)
    out = dict(n=n, V=V, H=H, C=C, B=B, epochs=epochs, cond_dim=cond_dim, k=k, lr=np.float64(lr), predict_seed=123,
               indptr=X.indptr.astype(np.int32), indices=X.indices.astype(np.int32),
               losses=np.asarray(losses[:n_fit], dtype=np.float64), pred=pred.astype(np.float32),
               topk=ref.evaluation.argtopk(masked, k)[1].astype(np.int64))
    if cond_dim:
        out["cond"] = cond
    for k_, v in init.items():
        out["init/" + k_] = v
    for k_, v in final.items():
        out["final/" + k_] = v
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "steps", n_fit, "first", losses[0], "last", losses[n_fit - 1])


def run_decoder_case(ref, name, n, V, H, D, B, epochs, dropout, data_seed=0, mean_len=6, k=10, lr=0.001):
    """aaerec/aae.py:461-584 (SURVEY 8(f)-3): the UNMODIFIED reference DecodingRecommender -- ``fit(condition_data, Y)``
    and ``predict(test_set)`` on a minimal Bags stand-in.  Per-step losses are captured by wrapping the module's
    ``F.binary_cross_entropy``."""
    aae = ref.aae
    Y = synth_sets(n, V, mean_len, min_len=2, seed=data_seed)
    cond = (np.random.RandomState(data_seed + 1).randn(n, D) * 0.5).astype(np.float32)
    conditions = _matrix_condition(ref, D)
    losses = []
    orig = aae.F.binary_cross_entropy

    def recording(*a, **kw):
        val = orig(*a, **kw)
        losses.append(float(val))
        return val

    class QueryBags(object):
        def __init__(self, rows):
            self.rows = rows

        def size(self, dim):
            return self.rows

        def get_attributes(self, keys):
            return [cond[: self.rows]]

        def tocsr(self):
            return Y[: self.rows]
    aae.F.binary_cross_entropy = recording
    try:
        torch.manual_seed(42)
        np.random.seed(42)
        rec = aae.DecodingRecommender(conditions, n_epochs=epochs, batch_size=B, n_hidden=H, lr=lr, verbose=False,
                                      dropout=dropout)
        # initial weights: replay the construction of Decoder(D, H, V) (aae.py:524-527) under the same seed
        st = torch.get_rng_state()
        dec0 = aae.Decoder(D, H, V, dropout=dropout)
        init = {k_: v.detach().cpu().numpy().copy() for k_, v in dec0.state_dict().items()}
        torch.set_rng_state(st)
        with contextlib.redirect_stdout(io.StringIO()):
            rec.fit([cond], Y)
        n_fit = len(losses)
        final = {k_: v.detach().cpu().numpy().copy() for k_, v in rec.mlp.state_dict().items()}
        with contextlib.redirect_stdout(io.StringIO()):
            pred = rec.predict(QueryBags(40))
    finally:
        aae.F.binary_cross_entropy = orig
    masked = ref.evaluation.remove_non_missing(pred, Y[:40].toarray(), copy=True)
    out = dict(n=n, V=V, H=H, D=D, B=B, epochs=epochs, dropout=np.asarray(dropout, dtype=np.float64), k=k,
               lr=np.float64(lr), indptr=Y.indptr.astype(np.int32), indices=Y.indices.astype(np.int32), cond=cond,
               losses=np.asarray(losses[:n_fit], dtype=np.float64), pred=pred.astype(np.float32),
               topk=ref.evaluation.argtopk(masked, k)[1].astype(np.int64))
    for k_, v in init.items():
        out["init/" + k_] = v
    for k_, v in final.items():
        out["final/" + k_] = v
    np.savez_compressed(os.path.join(GOLDEN, name + ".npz"), **out)
    print(name, "steps", n_fit, "first", losses[0], "last", losses[n_fit - 1])


def ranking_case(ref):
    rs = np.random.RandomState(7)
    Y = rs.rand(9, 64).astype(np.float32)
    Y[3, :] = 0.25                 # constant row: zero range
    Y[4, 10:20] = Y[4, 5]          # ties
    Xk = (rs.rand(9, 64) < 0.1).astype(np.float32)
    masked = ref.evaluation.remove_non_missing(Y, Xk, copy=True)
    cols5 = ref.evaluation.argtopk(masked, 5)[1]
    cols_all = ref.evaluation.argtopk(masked, None)[1]
    np.savez_compressed(os.path.join(GOLDEN, "ranking.npz"), Y=Y, Xk=Xk, masked=masked,
                        top5=cols5.astype(np.int64), full=cols_all.astype(np.int64))
    print("ranking ok")


def metrics_case(ref):
    """The reference's (mean, std) of every metric on the seeded case of tests/test_ranking_metrics.py, for
    test_oracle_metrics_match_reference where the reference package is absent."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_ranking_metrics import METRICS, reference_metrics
    want = np.asarray(reference_metrics(ref), dtype=np.float64)
    np.savez_compressed(os.path.join(GOLDEN, "metrics_reference.npz"), metrics=np.asarray(METRICS), want=want)
    print("metrics_reference ok")


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ref = load_reference()
    only = sys.argv[1] if len(sys.argv) > 1 else ""     # optional name prefix: regenerate a subset
    global run_case
    _run = run_case

    def run_case(ref_, name, **kw):
        if name.startswith(only):
            return _run(ref_, name, **kw)
    run_case(ref, "aae_small_dropout", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(.2, .2))
    run_case(ref, "aae_small_nodrop", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(0, 0))
    run_case(ref, "aae_small_cond", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(.2, .2), cond_dim=7)
    # the H=100 cases keep no initial weights (no test reads them; init_params rebuilds them from the seed): each
    # file stays under 1 MB
    run_case(ref, "aae_h100_dropout", n=96, V=520, H=100, C=50, B=32, epochs=2, dropout=(.2, .2), mean_len=8,
             store_init=False)
    # SURVEY 8(c) indicative configuration (losses + |W| sums only, weights rebuilt from the seed)
    run_case(ref, "aae_survey_nodrop", n=300, V=1000, H=100, C=50, B=100, epochs=1, dropout=(0, 0),
             mean_len=8, store_weights=False)
    run_case(ref, "aae_survey_dropout", n=300, V=1000, H=100, C=50, B=100, epochs=1, dropout=(.2, .2),
             mean_len=8, store_weights=False)
    # plain AutoEncoder (aae.py:221-458; AAERecommender(adversarial=False)): reconstruction phase only
    run_case(ref, "ae_small_dropout", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(.2, .2), adversarial=False)
    run_case(ref, "ae_h100_cond", n=96, V=520, H=100, C=50, B=32, epochs=2, dropout=(.2, .2), mean_len=8, cond_dim=7,
             adversarial=False, store_init=False)
    # non-default model options (pins the oracle only; the CUDA path is checked against the oracle in these modes by
    # tests/test_gpu_parity.py::test_edge_cases_empty_rows_unnormalized_prior_scale)
    run_case(ref, "aae_opts_unnorm_scale_lrs", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(.2, .2),
             model_kwargs=dict(normalize_inputs=False, prior_scale=0.5, gen_lr=0.002, reg_lr=0.0005))
    # DenoisingAutoEncoder (dae.py): zeros-noise corruption in front of the plain autoencoder step
    run_case(ref, "dae_small_dropout", n=130, V=257, H=24, C=10, B=50, epochs=2, dropout=(.2, .2), dae=True,
             model_kwargs=dict(noise_factor=0.3))
    run_case(ref, "dae_h100_cond", n=96, V=520, H=100, C=50, B=32, epochs=2, dropout=(.2, .2), mean_len=8, cond_dim=7,
             dae=True, store_init=False)
    # sibling models on the same decoder output layer (SURVEY 8(f)-3)
    if "vae_small".startswith(only):
        run_vae_case(ref, "vae_small", n=130, V=257, H=24, C=10, B=50, epochs=2)
    if "vae_h100_cond".startswith(only):
        run_vae_case(ref, "vae_h100_cond", n=96, V=520, H=100, C=50, B=32, epochs=2, mean_len=8, cond_dim=7)
    if "decoder_small_dropout".startswith(only):
        run_decoder_case(ref, "decoder_small_dropout", n=130, V=257, H=24, D=9, B=50, epochs=2, dropout=(.2, .2))
    if "decoder_h100_nodrop".startswith(only):
        run_decoder_case(ref, "decoder_h100_nodrop", n=96, V=520, H=100, D=30, B=32, epochs=2, dropout=(0, 0),
                         mean_len=8)
    if "ranking".startswith(only):
        ranking_case(ref)
    if "metrics_reference".startswith(only):
        metrics_case(ref)


if __name__ == "__main__":
    main()
