"""Shared helpers for the tests: golden loading and the oracle replay of a golden case."""
import os

import numpy as np
import scipy.sparse as sp
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

AAE_CASES = ["aae_small_dropout", "aae_small_nodrop", "aae_small_cond", "aae_h100_dropout",
             "aae_survey_nodrop", "aae_survey_dropout"]
AE_CASES = ["ae_small_dropout", "ae_h100_cond"]      # the plain AutoEncoder (AAERecommender(adversarial=False))
OPTION_CASES = ["aae_opts_unnorm_scale_lrs"]         # non-default normalize_inputs / prior_scale / learning rates
DAE_CASES = ["dae_small_dropout", "dae_h100_cond"]   # DenoisingAutoEncoder (dae.py; SURVEY 8(f)-3)


def load_case(name):
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    g["X"] = sp.csr_matrix((np.ones(len(g["indices"]), dtype=np.float32), g["indices"], g["indptr"]),
                           shape=(int(g["n"]), int(g["V"])))
    g["dropout"] = tuple(float(x) for x in g["dropout"])
    for k in ("n", "V", "H", "C", "B", "epochs", "cond_dim", "k"):
        g[k] = int(g[k])
    g["adversarial"] = bool(int(g.get("adversarial", 1)))
    g["dae"] = bool(int(g.get("dae", 0)))
    g["noise_factor"] = float(g.get("noise_factor", 0.2))
    g["normalize_inputs"] = bool(int(g.get("normalize_inputs", 1)))
    g["prior_scale"] = float(g.get("prior_scale", 0.0)) or None
    g["gen_lr"] = float(g.get("gen_lr", 0.001))
    g["reg_lr"] = float(g.get("reg_lr", 0.001))
    return g


def group(g, prefix):
    return {k[len(prefix) + 1:]: v for k, v in g.items() if k.startswith(prefix + "/")}


def oracle_replay(g, record_rng=False):
    """Run oracle/aae_oracle.py over a golden case exactly as the reference's fit loop does
    (aae.py:768-837): seed, build, shuffle per epoch, slice batches, three phases per batch."""
    from oracle import aae_oracle as O
    V, H, C, B = g["V"], g["H"], g["C"], g["B"]
    cond = g.get("cond")
    torch.manual_seed(42)
    np.random.seed(42)
    adv = g["adversarial"]
    params = O.init_params(V, H, C, C + g["cond_dim"], seed=None, adversarial=adv)
    if adv:
        model = O.OracleAAE(params, n_code=C, gen_lr=g["gen_lr"], reg_lr=g["reg_lr"],
                            normalize_inputs=g["normalize_inputs"])
    elif g["dae"]:
        model = O.OracleDAE(params, n_code=C, noise_factor=g["noise_factor"])
    else:
        model = O.OracleAE(params, n_code=C)
    X = g["X"]
    losses, rngs, batches = [], [], []
    for _ in range(g["epochs"]):
        perm = O.fit_epoch_order(X.shape[0])
        Xs = X[perm]
        cs = cond[perm] if cond is not None else None
        for s in range(0, X.shape[0], B):
            xb = Xs[s:s + B]
            cb = [cs[s:s + B]] if cs is not None else None
            if g["dae"]:
                rng = O.draw_dae_rng(xb.shape[0], V, H, C, g["dropout"])
            else:
                rng = O.draw_step_rng(xb.shape[0], H, C, g["dropout"], prior_scale=g["prior_scale"], adversarial=adv)
            losses.append(model.partial_fit(xb.toarray(), cb, rng))
            if record_rng:
                rngs.append(rng)
                batches.append((xb, cb))
    return model, np.asarray(losses), rngs, batches


def write_reference_standin(root):
    """A stand-in for the reference's ``aaerec`` package under ``root``: every module and name the import block of
    main.py:11-20 uses, as plain placeholders.  The overlay tests check which tree each name resolves to, which needs
    the tree's layout, not its code.  Returns ``root`` (the directory that contains ``aaerec/``)."""
    cls = "class %s(object):\n    pass\n"
    modules = {
        "__init__.py": "",
        "base.py": cls % "Recommender",
        "aae.py": "from .condition import ConditionList  # noqa: F401\nUSE_WANDB = True\n" + "".join(
            cls % c for c in ("Encoder", "Decoder", "Discriminator", "AutoEncoder", "AdversarialAutoEncoder",
                              "AAERecommender", "DecodingRecommender")),
        "dae.py": "def zeros_noise(x, p):\n    return x\n" + "".join(
            cls % c for c in ("DenoisingAutoEncoder", "DAERecommender")),
        "vae.py": "".join(cls % c for c in ("VAE", "VAERecommender")),
        "condition.py": "".join(cls % c for c in ("ConditionList", "PretrainedWordEmbeddingCondition",
                                                   "CategoricalCondition")),
        "datasets.py": cls % "Bags",
        "evaluation.py": cls % "Evaluation",
        "baselines.py": "".join(cls % c for c in ("RandomBaseline", "Countbased", "MostPopular")),
        "svd.py": cls % "SVDRecommender",
    }
    pkg = os.path.join(str(root), "aaerec")
    os.makedirs(pkg, exist_ok=True)
    for name, src in modules.items():
        with open(os.path.join(pkg, name), "w") as fh:
            fh.write(src)
    return str(root)


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ---- sibling models on the same decoder output layer (SURVEY 8(f)-3) -------------------------------------------------
VAE_CASES = ["vae_small", "vae_h100_cond"]                         # aaerec/vae.py
DECODER_CASES = ["decoder_small_dropout", "decoder_h100_nodrop"]   # DecodingRecommender, aaerec/aae.py:461-584


def load_sibling_case(name):
    g = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    g["X"] = sp.csr_matrix((np.ones(len(g["indices"]), dtype=np.float32), g["indices"], g["indptr"]),
                           shape=(int(g["n"]), int(g["V"])))
    for k in ("n", "V", "H", "C", "D", "B", "epochs", "cond_dim", "k", "predict_seed"):
        if k in g:
            g[k] = int(g[k])
    g["lr"] = float(g["lr"])
    if "dropout" in g:
        g["dropout"] = tuple(float(x) for x in g["dropout"])
    return g


def linear_init(shapes):
    """nn.Linear modules constructed in the given order on the CPU generator (stock init)."""
    p = {}
    for name, fin, fout in shapes:
        lin = torch.nn.Linear(fin, fout)
        p[name + ".weight"] = lin.weight.detach().clone()
        p[name + ".bias"] = lin.bias.detach().clone()
    return p


def oracle_replay_vae(g):
    """oracle.OracleVAE over a golden case as the reference runs it: VAE(...) construction under seed 42 (vae.py:76-87),
    fit (vae.py:188-229), then predict of the first 40 rows under ``predict_seed``."""
    from oracle import aae_oracle as O
    V, H, C, B, Dc = g["V"], g["H"], g["C"], g["B"], g["cond_dim"]
    cond = g.get("cond")
    torch.manual_seed(42)
    np.random.seed(42)
    params = linear_init([("fc1", V, H), ("fc21", H, C), ("fc22", H, C), ("fc3", C + Dc, H), ("fc4", H, V)])
    init = {k: v.clone() for k, v in params.items()}
    model = O.OracleVAE(params, n_code=C, lr=g["lr"])
    X = g["X"]
    losses, steps = [], []
    for _ in range(g["epochs"]):
        perm = O.fit_epoch_order(X.shape[0])
        Xs = X[perm]
        cs = cond[perm] if cond is not None else None
        for s in range(0, X.shape[0], B):
            xb = Xs[s:s + B]
            cb = [cs[s:s + B]] if cs is not None else None
            eps = torch.randn((xb.shape[0], C), dtype=torch.float32)       # vae.py:109 on the CPU generator
            losses.append(model.partial_fit(xb.toarray(), cb, eps))
            steps.append((xb, cb, eps))
    torch.manual_seed(g["predict_seed"])
    preds = []
    for s in range(0, 40, B):
        e = min(s + B, 40)
        eps = torch.randn((e - s, C), dtype=torch.float32)
        preds.append(model.predict(X[s:e].toarray(), [cond[s:e]] if cond is not None else None, eps))
    return model, np.asarray(losses), np.vstack(preds), init, steps


def oracle_replay_decoder(g):
    """oracle.OracleDecoder over a golden case as DecodingRecommender.fit runs it (aae.py:522-545)."""
    from oracle import aae_oracle as O
    V, H, D, B = g["V"], g["H"], g["D"], g["B"]
    cond = g["cond"]
    torch.manual_seed(42)
    np.random.seed(42)
    params = linear_init([("lin1", D, H), ("lin2", H, H), ("lin3", H, V)])
    init = {k: v.clone() for k, v in params.items()}
    model = O.OracleDecoder(params, lr=g["lr"])
    Y = g["X"]
    losses = []
    for _ in range(g["epochs"]):
        perm = O.fit_epoch_order(Y.shape[0])
        Ys, cs = Y[perm], cond[perm]
        for s in range(0, Y.shape[0], B):
            yb = Ys[s:s + B]
            b = yb.shape[0]
            masks = (O.draw_masks((b, H), g["dropout"][0], 1)[0], O.draw_masks((b, H), g["dropout"][1], 1)[0])
            losses.append(model.partial_fit([cs[s:s + B]], yb.toarray(), {"ae_dec": masks}))
    pred = np.vstack([model.predict([cond[s:min(s + B, 40)]]) for s in range(0, 40, B)])
    return model, np.asarray(losses), pred, init
