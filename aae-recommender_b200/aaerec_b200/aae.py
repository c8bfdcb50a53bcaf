"""B200-native Adversarial Autoencoder recommender behind the reference's own API.

Mirrors ``aaerec/aae.py``: ``AdversarialAutoEncoder`` (589-870; same constructor kwargs and
defaults, ``fit`` / ``partial_fit`` / ``predict`` / ``eval`` / ``train`` / ``__str__``) and
``AAERecommender`` (873-977; ``train(training_set)`` / ``predict(test_set)``), so that
``main.py`` / ``eval/*.py`` can construct it unchanged.  All numerics run in the CUDA kernels of
``libaae_b200.so`` through :class:`aaerec_b200.engine.AAEEngine`; there is no PyTorch/CPU fallback.

Additions that are not in the reference (defaults keep the reference's behaviour):
  ``predict_topk(X, k)``  fused predict + remove_non_missing + argtopk without the dense [n,V] matrix
  ``evaluate_topk(X, Y, metrics)``  the harness' ranking metrics (evaluation.py:70-164, 202-240) on the device
  ``items=`` / ``exclude=``  candidate restriction of both: only eligible, non-excluded items are ranked
  ``rng='native'|'oracle'``  in-kernel Philox dropout / prior sampling, or the reference's CPU-generator
                           draws in the reference's order (bit-identical masks; used by parity tests)
  ``impl``  decoder-output kernel: 'auto', 'simt' (exact fp32 CUDA cores), 'tc' = 'parity' (tcgen05 3xTF32, fp32-accurate),
            'tf32' = 'fast' (single-pass TF32: ~1e-3 relative logits, outside the parity gates)
  ``device`` / ``rank`` / ``world``  item-sharded multi-GPU
"""
import numpy as np
import scipy.sparse as sp
import torch

from .base import Recommender
from .condition import _check_conditions, CondAdapter
from .engine import AAEEngine
from .filters import RankFilter

torch.manual_seed(42)   # aae.py:27 -- the reference seeds the CPU generator at import
TINY = 1e-12
STATUS_FORMAT = "[ R: {:.4f} | D: {:.4f} | G: {:.4f} ]"


def log_losses(*losses):
    print('\r' + STATUS_FORMAT.format(*losses), end='', flush=True)


PRIOR_ACTIVATIONS = {'categorical': 'softmax', 'bernoulli': 'sigmoid', 'gauss': 'linear'}
SUPPORTED_OPTIMIZERS = {'adam'}   # the reference's table also has 'sgd' (aae.py:216-219)


def _init_linear_params(n_items, n_hidden, n_code, code_size, adversarial=True):
    """Same construction order and stock nn.Linear init as aae.py:782-792, on the CPU generator.  The plain
    AutoEncoder builds no discriminator (aae.py:368-387) and so draws nothing for it."""
    out = {}
    for name, fin, fout in (
            ("enc.lin1", n_items, n_hidden), ("enc.lin2", n_hidden, n_hidden), ("enc.lin3", n_hidden, n_code),
            ("dec.lin1", code_size, n_hidden), ("dec.lin2", n_hidden, n_hidden), ("dec.lin3", n_hidden, n_items),
            ("disc.lin1", n_code, n_hidden), ("disc.lin2", n_hidden, n_hidden), ("disc.lin3", n_hidden, 1)):
        if name.startswith("disc") and not adversarial:
            out[name + ".weight"] = torch.zeros(fout, fin)
            out[name + ".bias"] = torch.zeros(fout)
            continue
        lin = torch.nn.Linear(fin, fout)
        out[name + ".weight"] = lin.weight.detach()
        out[name + ".bias"] = lin.bias.detach()
    return out


def _draw_step_rng(B, n_hidden, n_code, dropout, prior_scale, adversarial=True):
    """The reference's draws for one partial_fit, same calls in the same order on torch's global CPU
    generator (SURVEY 8(a) A11): nn.Dropout == x * empty_like(x).bernoulli_(1-p).div_(1-p); p == 0 draws
    nothing; z_real = torch.randn (aae.py:716)."""
    p1, p2 = dropout

    def mask(p):
        if p == 0:
            return None
        return torch.empty((B, n_hidden), dtype=torch.float32).bernoulli_(1 - p).div_(1 - p)

    def pair():
        return (mask(p1), mask(p2))
    r = {"ae_enc": pair(), "ae_dec": pair()}
    if not adversarial:       # AutoEncoder.ae_step draws the four reconstruction-phase masks only (aae.py:267-306)
        return r
    z = torch.randn((B, n_code))
    if prior_scale is not None:
        z = z * prior_scale
    r["z_real"] = z
    r["disc_real"] = pair()
    r["disc_fake"] = pair()
    r["gen_enc"] = pair()
    r["gen_disc"] = pair()
    return r


class _LinearView(object):
    def __init__(self, weight, bias):
        self.weight, self.bias = weight, bias
        self.in_features, self.out_features = weight.shape[1], weight.shape[0]


class _ModuleView(object):
    """Read-only view of a module's weights in the reference's layout (``.lin1.weight`` ...)."""

    def __init__(self, sd, prefix):
        self._sd = {k[len(prefix) + 1:]: v for k, v in sd.items() if k.startswith(prefix + ".")}
        for i in (1, 2, 3):
            setattr(self, "lin%d" % i, _LinearView(self._sd["lin%d.weight" % i], self._sd["lin%d.bias" % i]))

    def state_dict(self):
        return dict(self._sd)


def _canonical_csr(X, what="input"):
    """Any 2-D batch (dense ndarray as the reference passes to partial_fit, or scipy sparse) -> CSR with duplicates
    summed, explicit zeros dropped and sorted column indices.  The kernels train on *binary* sets (indptr/indices
    only): the reference's BCE rejects targets outside [0,1] (``RuntimeError``, SURVEY 8(b)), and fractional values,
    which the reference would use as soft targets, are outside the accelerated envelope."""
    if not sp.issparse(X):
        X = sp.csr_matrix(np.asarray(X))
    X = X.tocsr()
    if not X.has_canonical_format:
        X = X.copy()
        X.sum_duplicates()
    if X.nnz and (X.data == 0).any():
        X = X.copy()
        X.eliminate_zeros()
    if not X.has_sorted_indices:
        X = X.sorted_indices()
    if X.nnz:
        if X.data.max() > 1 or X.data.min() < 0:
            raise RuntimeError("all elements of target should be between 0 and 1")
        if (X.data != 1).any():
            raise NotImplementedError("%s has fractional entries: the accelerated path handles binary item sets only"
                                      % what)
    return X


class _OptimView(object):
    """Read-only stand-in for the reference's ``torch.optim.Adam`` attributes (``enc_optim`` ... aae.py:798-804):
    hyper-parameters in ``param_groups`` and the Adam moments in ``state_dict()`` (torch's key names)."""

    def __init__(self, model, which, lr):
        self._model, self._which = model, which
        self.param_groups = [{"lr": lr, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0, "amsgrad": False}]
        self.defaults = dict(self.param_groups[0])

    def state_dict(self):
        eng = self._model.engine
        state = {}
        if eng is not None:
            for name, (m, v) in eng.optim_state(self._which).items():
                state[name] = {"step": eng.steps_done, "exp_avg": m, "exp_avg_sq": v}
        return {"state": state, "param_groups": [dict(self.param_groups[0])]}

    def zero_grad(self):
        """Gradients never persist between kernels."""

    def step(self):
        raise NotImplementedError("the optimizer updates are fused into the step kernels; call partial_fit or the "
                                  "phase methods ae_step / disc_step / gen_step")


class AdversarialAutoEncoder(object):
    """ Adversarial Autoencoder (aae.py:589) """
    adversarial = True
    _announce = True       # fit() prints the reference's "Using condition, code size" line (aae.py:776-780)

    def _log_losses(self, losses):
        log_losses(*losses)

    def __init__(self,
                 n_hidden=100,
                 n_code=50,
                 gen_lr=0.001,
                 reg_lr=0.001,
                 prior='gauss',
                 prior_scale=None,
                 batch_size=100,
                 n_epochs=500,
                 optimizer='adam',
                 normalize_inputs=True,
                 activation='ReLU',
                 dropout=(.2, .2),
                 conditions=None,
                 verbose=True,
                 rng='native',
                 impl='auto',
                 device=None,
                 rank=0,
                 world=1,
                 group=None,
                 seed=0,
                 use_graph=True):
        self.prior = prior.lower()
        self.prior_scale = prior_scale
        self.encoder_activation = PRIOR_ACTIVATIONS[self.prior]   # KeyError on unknown prior, as aae.py:612-613
        self.optimizer = optimizer.lower()
        self.n_hidden = n_hidden
        self.n_code = n_code
        self.gen_lr, self.reg_lr = gen_lr, reg_lr
        self.batch_size = batch_size
        self.verbose = verbose
        self.n_epochs = n_epochs
        self.normalize_inputs = normalize_inputs
        self.dropout = dropout
        self.activation = activation
        self.conditions = conditions
        self.rng = rng
        self.impl = impl
        self.device, self.rank, self.world, self.group = device, rank, world, group
        self.seed = seed
        self.use_graph = use_graph
        self.engine = None
        self._adapter = None
        self._mode_train = True
        self.predict_batch_size = 1024   # query rows per launch of predict_topk (>= batch_size)
        self.record_losses = False   # True: keep every step's (R, D, G) in .loss_history (forces a sync per step)
        self.last_losses = None
        # supported envelope (SURVEY 8(b)); everything else fails loudly, there is no fallback path
        if self.prior != 'gauss':
            raise NotImplementedError("accelerated path supports prior='gauss' only (got %r)" % prior)
        if activation != 'ReLU':
            raise NotImplementedError("accelerated path supports activation='ReLU' only (got %r)" % activation)
        if self.optimizer not in SUPPORTED_OPTIMIZERS:
            if self.optimizer == 'sgd':
                raise NotImplementedError("accelerated path supports optimizer='adam' only")
            raise KeyError(optimizer)
        if rng not in ('native', 'oracle'):
            raise ValueError("rng must be 'native' or 'oracle'")
        # aae.py:798-804: enc_optim and dec_optim at gen_lr, gen_optim and disc_optim at reg_lr
        self.enc_optim = _OptimView(self, "enc", gen_lr)
        self.dec_optim = _OptimView(self, "dec", gen_lr)
        if self.adversarial:
            self.gen_optim = _OptimView(self, "gen", reg_lr)
            self.disc_optim = _OptimView(self, "disc", reg_lr)

    def __str__(self):
        desc = "Adversarial Autoencoder"
        n_h, n_c = self.n_hidden, self.n_code
        gen, reg = self.gen_lr, self.reg_lr
        desc += " ({}, {}, {}, {}, {})".format(n_h, n_h, n_c, n_h, n_h)
        desc += " optimized by " + self.optimizer
        desc += " with learning rates Gen, Reg = {}, {}".format(gen, reg)
        desc += ", using a batch size of {}".format(self.batch_size)
        desc += "\nMatching the {} distribution".format(self.prior)
        desc += " by {} activation.".format(self.encoder_activation)
        if self.conditions:
            desc += "\nConditioned on " + ', '.join(self.conditions.keys())
        return desc

    # -- mode switches (dropout is decided per kernel call; kept for API compatibility, aae.py:636-660)
    def eval(self):
        self._mode_train = False
        if self.conditions:
            self.conditions.eval()

    def train(self):
        self._mode_train = True
        if self.conditions:
            self.conditions.train()

    def zero_grad(self):
        """Gradients never persist between kernels; nothing to clear."""

    # -- weights in the reference's layout
    @property
    def enc(self):
        return _ModuleView(self.engine.state_dict(), "enc") if self.engine else None

    @property
    def dec(self):
        return _ModuleView(self.engine.state_dict(), "dec") if self.engine else None

    @property
    def disc(self):
        return _ModuleView(self.engine.state_dict(), "disc") if self.engine else None

    def state_dict(self):
        return self.engine.state_dict()

    # -- helpers
    def _build(self, n_items, code_size, params=None):
        if params is None:
            params = _init_linear_params(n_items, self.n_hidden, self.n_code, code_size, self.adversarial)
        self.engine = AAEEngine(n_items, self.n_hidden, self.n_code, cond_dim=code_size - self.n_code,
                                gen_lr=self.gen_lr, reg_lr=self.reg_lr, dropout=self.dropout,
                                prior_scale=self.prior_scale, normalize_inputs=self.normalize_inputs,
                                device=self.device, rank=self.rank, world=self.world, group=self.group,
                                impl=self.impl, seed=self.seed, max_batch=self.batch_size,
                                use_graph=self.use_graph, adversarial=self.adversarial)
        self.engine.load_params(params)
        self.last_losses = None

    def _cond_adapter(self):
        if not self.conditions:
            return None
        if self._adapter is None or self._adapter.conditions is not self.conditions:
            self._adapter = CondAdapter(self.conditions)
        return self._adapter

    @staticmethod
    def _csr_batch(X):
        X = _canonical_csr(X, "batch")
        return X.indptr.astype(np.int32, copy=False), X.indices.astype(np.int32, copy=False)

    def _draws(self, B):
        if self.rng != 'oracle':
            return None
        return _draw_step_rng(B, self.n_hidden, self.n_code, self.dropout, self.prior_scale, self.adversarial)

    # -- condition plumbing of one training batch
    def _cond_begin(self, cond_batch, B):
        """Before the step: row conditions hand over their float rows (host), generic ones are encoded through their
        own protocol after ``conditions.zero_grad()`` (aae.py:698-700).  Returns (host rows or None, autograd leaves)."""
        ad = self._cond_adapter()
        if ad is None or cond_batch is None:
            return None, None
        if ad.all_rows:
            return ad.encode_all_rows(cond_batch), None
        self.conditions.zero_grad()
        rows_dev, leaves = ad.encode_batch(cond_batch, self.engine.dev, want_grad=True)
        self.engine.set_cond_rows(rows_dev, B)
        if leaves:
            self.engine.snapshot_dec_lin1()
        return None, leaves

    def _cond_end(self, leaves, B):
        """After the reconstruction phase: the conditions' backward and ``conditions.step()`` (aae.py:703-709)."""
        if leaves is None:
            return
        ad = self._cond_adapter()
        ad.backward_and_step(leaves, self.engine.cond_grad(B) if leaves else None)

    # -- training
    def partial_fit(self, X, y=None, condition_data=None, step=None):
        """ Performs reconstrction, discimination, generator training steps (aae.py:745-766) """
        if y is not None:
            raise NotImplementedError("(Semi-)supervised usage not supported")
        use_condition = _check_conditions(self.conditions, condition_data)
        if self.engine is None:
            code_size = self.n_code + (self.conditions.size_increment() if use_condition else 0)
            self._build(X.shape[1], code_size)
        indptr, indices = self._csr_batch(X)
        B = int(indptr.shape[0]) - 1
        self.train()
        rows, leaves = self._cond_begin(condition_data if use_condition else None, B)
        draws = self._draws(B)
        self.engine.train_step_host(indptr, indices, rows, injected=draws is not None, rng_draws=draws,
                                    cond_on_device=leaves is not None)
        self._cond_end(leaves, B)
        if self.verbose:
            self._log_losses(self.losses())
        return self

    def _phase(self, phase, batch, condition_data):
        """One of the reference's three phase methods (aae.py:676-743) on its own: same argument (the batch; a dense
        tensor/ndarray as the reference passes, or scipy sparse), same return value (the phase's loss as float)."""
        if torch.is_tensor(batch):
            batch = batch.detach().cpu().numpy()
        eng = self.engine
        if phase == "ae":
            use_condition = _check_conditions(self.conditions, condition_data)
            if eng is None:
                code_size = self.n_code + (self.conditions.size_increment() if use_condition else 0)
                self._build(batch.shape[1], code_size)
                eng = self.engine
            indptr, indices = self._csr_batch(batch)
            B = int(indptr.shape[0]) - 1
            rows, leaves = self._cond_begin(condition_data if use_condition else None, B)
            eng.upload_csr(indptr, indices, rows)
            self._phase_B = B
            draws = self._draws(B)
            if draws is not None:
                eng.set_rng_draws(B, draws)
            self._phase_injected = draws is not None
            loss = eng.phase_step("ae", B, self._phase_injected)
            self._cond_end(leaves, B)
            return loss
        if eng is None:
            raise RuntimeError("%s_step before ae_step: the model is built by the first reconstruction step" % phase)
        return eng.phase_step(phase, self._phase_B, self._phase_injected)

    def ae_step(self, batch, condition_data=None):
        """aae.py:676-711.  The four optimizers share one Adam step counter, so the three phase methods must be
        called in partial_fit's order (ae_step, disc_step, gen_step on the same batch)."""
        return self._phase("ae", batch, condition_data)

    def disc_step(self, batch):
        """aae.py:713-732 (on the batch ae_step saw)."""
        return self._phase("disc", batch, None)

    def gen_step(self, batch):
        """aae.py:734-743 (on the batch ae_step saw)."""
        return self._phase("gen", batch, None)

    def losses(self):
        """(recon, disc, gen) losses of the last step -- a device->host read (synchronises)."""
        self.last_losses = tuple(float(x) for x in self.engine.losses.cpu().tolist())
        self.engine.check_exchange()
        return self.last_losses

    def fit(self, X, y=None, condition_data=None):
        """aae.py:768-837: build, then per epoch shuffle and walk the batches.  The training matrix (and the matrix of
        row conditions) is uploaded once; every epoch the host draws the reference's permutation and the batches are
        assembled on the device (``aae_batch_gather``)."""
        if y is not None:
            raise NotImplementedError("(Semi-)supervised usage not supported")
        use_condition = _check_conditions(self.conditions, condition_data)
        if use_condition:
            code_size = self.n_code + self.conditions.size_increment()
            if self._announce:
                print(("" if self.adversarial else "[ae] ") + "Using condition, code size:", code_size)
        else:
            code_size = self.n_code
            if self._announce:
                print(("" if self.adversarial else "[ae] ") + "Not using condition, code size:", code_size)
        X = _canonical_csr(X, "training matrix")
        self._build(X.shape[1], code_size)
        eng = self.engine
        ad = self._cond_adapter() if use_condition else None
        cond_all = ad.encode_all_rows(condition_data) if (ad is not None and ad.all_rows) else None
        eng.set_epoch_data(X.indptr, X.indices, cond_all)
        n = X.shape[0]
        self.loss_history = []
        self.epoch_seconds = []          # wall-clock of every epoch (one synchronisation per epoch)
        self.train()
        import time
        for epoch in range(self.n_epochs):
            t_epoch = time.perf_counter()
            if self.verbose:
                print("Epoch", epoch + 1)
            # sklearn.utils.shuffle(X, *condition_data) with random_state=None permutes arange(n) with the
            # global numpy generator (aae.py:815-817); same stream consumption here.
            perm = np.arange(n)
            np.random.shuffle(perm)
            eng.set_epoch_perm(perm)
            for start in range(0, n, self.batch_size):
                end = min(start + self.batch_size, n)
                B = end - start
                leaves = None
                if ad is not None and not ad.all_rows:
                    rows = perm[start:end]
                    _, leaves = self._cond_begin([ad.take(c, rows) for c in condition_data], B)
                eng.gather_batch(start, B)
                if getattr(self, "_fit_step", None) is not None:     # DenoisingAutoEncoder: corruption + step
                    self._fit_step(B, leaves)
                else:
                    draws = self._draws(B)
                    if draws is not None:
                        eng.set_rng_draws(B, draws)      # oracle RNG: masks (none when p == 0) and the prior sample
                    eng.train_step(B, draws is not None)
                    self._cond_end(leaves, B)
                if self.verbose or self.record_losses:
                    cur = self.losses()
                    if self.record_losses:
                        self.loss_history.append(cur)
                    if self.verbose:
                        self._log_losses(cur)
            if self.verbose:
                print()
            torch.cuda.synchronize(eng.dev)
            self.epoch_seconds.append(time.perf_counter() - t_epoch)
        eng.check_exchange()
        return self

    # -- prediction
    def _iter_batches(self, X, condition_data, batch_size=None):
        """Query batches of an eval-mode pass: the query matrix (and row-condition matrix) is uploaded once and the
        batches are built on the device; generic conditions are encoded per batch through their protocol."""
        batch_size = batch_size or self.batch_size
        use_condition = _check_conditions(self.conditions, condition_data)
        self.eval()
        X = _canonical_csr(X, "query matrix")
        eng = self.engine
        ad = self._cond_adapter() if use_condition else None
        cond_all = ad.encode_all_rows(condition_data) if (ad is not None and ad.all_rows) else None
        eng.set_epoch_data(X.indptr, X.indices, cond_all)
        eng.set_epoch_perm(None)
        n = X.shape[0]
        for start in range(0, n, batch_size):
            end = min(start + batch_size, n)
            B = end - start
            eng.gather_batch(start, B)
            if ad is not None and not ad.all_rows:
                rows = np.arange(start, end)
                with torch.no_grad():
                    rows_dev, _ = ad.encode_batch([ad.take(c, rows) for c in condition_data], eng.dev, want_grad=False)
                eng.set_cond_rows(rows_dev, B)
            yield start, end, B

    def predict(self, X, condition_data=None):
        """aae.py:840-870: dense float32 [n, n_items] sigmoid probabilities (API-compatible; for
        million-item vocabularies use predict_topk)."""
        eng = self.engine
        n = X.shape[0]
        out = np.empty((n, eng.V), dtype=np.float32)
        dev = torch.empty(self.batch_size, eng.Vloc, dtype=torch.float32, device=eng.dev)
        for start, end, B in self._iter_batches(X, condition_data):
            eng.scores(B, dev, apply_sigmoid=True)
            if eng.world == 1:
                out[start:end] = dev[:B].cpu().numpy()
            else:
                out[start:end] = eng._gather_items(dev[:B].t().contiguous()).t().cpu().numpy()
        eng.check_exchange()
        return out

    def predict_topk(self, X, k, condition_data=None, mask_known=True, return_scores=False, shard="items",
                     items=None, exclude=None):
        """Top-k unknown items per row = argtopk(remove_non_missing(predict(X), X), k)[1]
        (evaluation.py:183-199, 20-58) without materialising [n, n_items] on the host.

        Multi-GPU: ``shard='items'`` ranks every query against the local item shard and merges the per-shard lists
        (one all-gather per batch); ``shard='sets'`` gives every rank a full-weight replica (built once) and its own
        slice of the query rows -- no communication in the query loop; the slices are exchanged at the end.

        Candidate restriction (both absent: the unrestricted ranking above):
          ``items``   eligible items: 1-D array of item ids in [0, n_items) (duplicates allowed) or a boolean mask of
                      length n_items (a block list is ``items=~blocked``); only these are ranked.
          ``exclude`` scipy sparse [n, n_items]: the nonzero entries of row i are never returned for row i.
        Semantics: ineligible items and excluded (row, item) pairs are never returned.  With ``mask_known`` a known
        item that is eligible and not excluded ranks below every unknown one (score -FLT_MAX, as without a filter); a
        known item that is ineligible or excluded is not returned.  Ties go to the lower item id.  A row with fewer
        than k returnable items is padded at the end with item id -1 and score -inf.  ``k=None`` (or k > MAX_TOPK)
        gives the full ranking of the eligible items: A columns for k=None (A = number of eligible items), min(k, A)
        otherwise, padded the same way; item-sharded full rankings raise as without a filter.  Ids out of range, a mask of the wrong length or an ``exclude`` of the wrong
        shape raise ValueError.  The eligible rows of the output layer are ranked as a compact copy cached on the
        engine (rebuilt when the eligible set or the weights change)."""
        filt = RankFilter.build(self.engine.V, X.shape[0], items, exclude)
        if k is None or k > self.MAX_TOPK:
            # argtopk's k=None / k >= size branch (evaluation.py:48-52): the full ranking of every row
            return self._full_ranking(X, eng_k=k, condition_data=condition_data, mask_known=mask_known,
                                      return_scores=return_scores, filt=filt)
        if shard == "sets" and self.engine.world > 1:
            return self._predict_topk_set_sharded(X, k, condition_data, mask_known, return_scores, filt)
        eng = self.engine
        n = X.shape[0]
        kk = min(k, eng.V)
        idx = np.empty((n, kk), dtype=np.int64)
        val = np.empty((n, kk), dtype=np.float32) if return_scores else None
        # rows are independent in eval mode: rank in query batches of >= 1024 rows whatever the training batch size
        # (the fused path keeps no [B,V] matrix, so the batch only sizes the candidate lists)
        pb = max(self.batch_size, self.predict_batch_size)
        for start, end, B in self._iter_batches(X, condition_data, batch_size=pb):
            i, v = eng.topk(B, kk, mask_known=mask_known, filt=None if filt is None else filt.rows(start, end))
            idx[start:end] = i.cpu().numpy()
            if return_scores:
                val[start:end] = v.cpu().numpy()
        eng.check_exchange()
        return (idx, val) if return_scores else idx



    MAX_TOPK = 4096       # envelope of the selection kernels (aae_masked_topk / aae_predict_topk2)

    def _full_ranking(self, X, eng_k, condition_data, mask_known, return_scores, filt=None):
        """All items of every row in descending order of remove_non_missing(predict(X), X) -- ``argtopk(.., k=None)``
        (evaluation.py:48-52), or its first ``k`` columns for a k beyond the selection kernels' envelope.  The [B, V]
        logit matrix is built by the decoder kernel and sorted on the device (known items last, ties by lower item id);
        this is the unbounded-metric convenience path, not the hot path: MRR / MAP over the whole vocabulary come from
        ``evaluate_topk`` (rank counts), which never sorts."""
        eng = self.engine
        if eng.world > 1:
            raise NotImplementedError("full rankings (k=None or k > %d) on item shards: use evaluate_topk for unbounded "
                                      "metrics, or a single-GPU / set-sharded replica" % self.MAX_TOPK)
        if filt is not None:
            return self._full_ranking_filtered(X, eng_k, condition_data, mask_known, return_scores, filt)
        n, V = X.shape[0], eng.V
        kk = V if eng_k is None else min(eng_k, V)
        idx = np.empty((n, kk), dtype=np.int64)
        val = np.empty((n, kk), dtype=np.float32) if return_scores else None
        dev = torch.empty(self.batch_size, V, dtype=torch.float32, device=eng.dev)
        for start, end, B in self._iter_batches(X, condition_data):
            eng.scores(B, dev, apply_sigmoid=False)
            sc = dev[:B]
            if mask_known:
                ip = eng.indptr[:B + 1].long()
                cols = eng.indices[:int(ip[-1])].long()
                rows = torch.repeat_interleave(torch.arange(B, device=eng.dev), ip[1:] - ip[:-1])
                sc[rows, cols] = -float("inf")
            v, i = torch.sort(sc, dim=1, descending=True, stable=True)
            idx[start:end] = i[:, :kk].cpu().numpy()
            if return_scores:
                val[start:end] = v[:, :kk].cpu().numpy()
        return (idx, val) if return_scores else idx

    def _full_ranking_filtered(self, X, eng_k, condition_data, mask_known, return_scores, filt):
        """``_full_ranking`` under a candidate filter: the [B, A] logits of the eligible items only (compact copy of
        the output layer) are sorted on the device and mapped back to item ids; known items score -FLT_MAX (below
        every unknown one), excluded ones -inf, which come out as the (-1, -inf) padding at the end of the row."""
        eng = self.engine
        n, V = X.shape[0], eng.V
        A = filt.n_eligible(V)
        kk = A if eng_k is None else min(eng_k, A)
        idx = np.empty((n, kk), dtype=np.int64)
        val = np.empty((n, kk), dtype=np.float32) if return_scores else None
        for start, end, B in self._iter_batches(X, condition_data):
            if filt.items is None:
                sc = eng.scores(B, torch.empty(B, V, dtype=torch.float32, device=eng.dev), apply_sigmoid=False)
                ids = torch.arange(V, dtype=torch.int32, device=eng.dev)
            else:
                sc, ids = eng.compact_scores(B, filt.items)
            ids = ids.long()

            def fill(indptr, indices, value):
                ip = torch.as_tensor(np.asarray(indptr, dtype=np.int64), device=eng.dev)
                g = torch.as_tensor(np.asarray(indices, dtype=np.int64), device=eng.dev)[: int(ip[-1])]
                rows = torch.repeat_interleave(torch.arange(B, device=eng.dev), ip[1:] - ip[:-1])
                col = torch.searchsorted(ids, g).clamp_(max=max(A - 1, 0))
                hit = ids[col] == g if A else torch.zeros_like(g, dtype=torch.bool)
                sc[rows[hit], col[hit]] = value
            if mask_known:
                fill(eng.indptr[:B + 1].cpu().numpy(), eng.indices[:int(eng.indptr[B])].cpu().numpy(),
                     -float(np.finfo(np.float32).max))
            if filt.exclude is not None:
                ex = filt.exclude[start:end]
                fill(ex.indptr, ex.indices, -float("inf"))
            v, i = torch.sort(sc, dim=1, descending=True, stable=True)
            v, i = v[:, :kk], ids[i[:, :kk]]
            i.masked_fill_(v == -float("inf"), -1)
            idx[start:end] = i.cpu().numpy()
            if return_scores:
                val[start:end] = v.cpu().numpy()
        return (idx, val) if return_scores else idx

    def _predict_topk_set_sharded(self, X, k, condition_data, mask_known, return_scores, filt=None):
        import torch.distributed as dist
        eng = self.engine
        if getattr(self, "_replica", None) is None or self._replica_step != eng.steps_done:
            self._replica = eng.make_replica(max_batch=max(self.batch_size, self.predict_batch_size))   # collective
            self._replica_step = eng.steps_done
        n = X.shape[0]
        per = (n + eng.world - 1) // eng.world
        lo, hi = min(n, eng.rank * per), min(n, (eng.rank + 1) * per)
        Xl = _canonical_csr(X, "query matrix")[lo:hi]
        cl = None
        if condition_data is not None:
            ad = self._cond_adapter()
            cl = [ad.take(c, np.arange(lo, hi)) for c in condition_data]
        main, self.engine = self.engine, self._replica
        fkw = {} if filt is None else dict(items=filt.items,
                                           exclude=None if filt.exclude is None else filt.exclude[lo:hi])
        try:
            out = self.predict_topk(Xl, k, condition_data=cl, mask_known=mask_known, return_scores=return_scores,
                                    **fkw) \
                if hi > lo else ((np.zeros((0, min(k, eng.V)), np.int64), np.zeros((0, min(k, eng.V)), np.float32))
                                 if return_scores else np.zeros((0, min(k, eng.V)), np.int64))
        finally:
            self.engine = main
        parts = [None] * eng.world
        dist.all_gather_object(parts, out, group=eng.group)
        if return_scores:
            return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])
        return np.concatenate(parts)

    def gold_ranks(self, X, Y, condition_data=None, batch_size=256, items=None, exclude=None):
        """Rank (1-based) of every held-out item of ``Y`` (scipy sparse [n, n_items], the harness' ``y_test``) in the
        ranking of remove_non_missing(predict(X), X): (indptr, ranks) aligned with ``Y.tocsr()``'s entries.  The score
        matrix is built and ranked on the device batch by batch; only the ranks travel to the host.

        ``items`` / ``exclude`` (as in ``predict_topk``, same ValueErrors): the ranks are the 1-based positions in
        the list ``predict_topk(X, None, items=items, exclude=exclude)`` returns.  A gold item that is ineligible or
        excluded for its row is not in that list: its rank is 0."""
        filt = RankFilter.build(self.engine.V, X.shape[0], items, exclude)
        return self._gold_ranks(X, Y, condition_data, batch_size, filt)

    def _gold_ranks(self, X, Y, condition_data, batch_size, filt):
        eng = self.engine
        Y = _canonical_csr(Y, "gold matrix")
        if Y.shape != (X.shape[0], eng.V):
            raise ValueError("gold matrix has shape %s, expected (%d, %d)" % (Y.shape, X.shape[0], eng.V))
        ranks = np.zeros(Y.nnz, dtype=np.int64)
        # returnable gold only go to the device; the others keep rank 0
        keep = None if filt is None else filt.returnable(Y.indptr, Y.indices)
        scratch = torch.empty(min(batch_size, X.shape[0]), eng.Vloc, dtype=torch.float32, device=eng.dev)
        for start, end, B in self._iter_batches(X, condition_data, batch_size=batch_size):
            lo, hi = int(Y.indptr[start]), int(Y.indptr[end])
            if keep is None:
                gp = (Y.indptr[start:end + 1] - lo).astype(np.int32)
                ranks[lo:hi] = eng.gold_ranks(B, gp, Y.indices[lo:hi], scratch=scratch)
                continue
            m = keep[lo:hi]
            gp = np.concatenate(([0], np.cumsum(m)))[Y.indptr[start:end + 1] - lo].astype(np.int32)
            ranks[lo:hi][m] = eng.gold_ranks(B, gp, Y.indices[lo:hi][m], scratch=scratch,
                                             filt=filt.rows(start, end))
        eng.check_exchange()
        return Y.indptr.astype(np.int64), ranks

    def evaluate_topk(self, X, Y, metrics, condition_data=None, batch_size=256, items=None, exclude=None):
        """The harness' ``evaluate(y_test, remove_non_missing(predict(X), X), metrics)`` (evaluation.py:202-240, 395)
        without the dense [n, n_items] matrix ever reaching the host: [(mean, std)] per metric.  ``metrics``: keys of
        evaluation.py:166-180 ('mrr@5', 'map', 'P@1' ...) or the reference's metric objects.

        ``items`` / ``exclude`` (as in ``predict_topk``): the same metrics of the list ``predict_topk(X, None,
        items=items, exclude=exclude)`` returns.  A gold item that is ineligible or excluded for its row is never a
        hit and takes no place in MAP's count; a row whose gold are all such scores 0.  ``P`` without k divides by the
        number of eligible items (the list's length)."""
        from .ranking import metrics_from_ranks
        filt = RankFilter.build(self.engine.V, X.shape[0], items, exclude)
        indptr, ranks = self._gold_ranks(X, Y, condition_data, batch_size, filt)
        V = self.engine.V
        return metrics_from_ranks(indptr, ranks, metrics, V if filt is None else filt.n_eligible(V))


class AutoEncoder(AdversarialAutoEncoder):
    """Plain (non-adversarial) autoencoder, aae.py:221-458: the reconstruction phase of the AAE alone, enc_optim
    and dec_optim both at ``lr`` (aae.py:393-394), no discriminator, no prior.  Same kernels, same engine with the
    adversarial phases switched off; the losses read (R, 0, 0) as the reference logs them (aae.py:341-342)."""
    adversarial = False

    def __init__(self, n_hidden=100, n_code=50, lr=0.001, batch_size=100, n_epochs=500, optimizer='adam',
                 normalize_inputs=True, activation='ReLU', dropout=(.2, .2), conditions=None, verbose=True,
                 rng='native', impl='auto', device=None, rank=0, world=1, group=None, seed=0, use_graph=True):
        # reg_lr = 0: the second Adam state of enc.lin1 (gen_optim in the AAE) is never stepped and stays exactly zero
        super().__init__(n_hidden=n_hidden, n_code=n_code, gen_lr=lr, reg_lr=0.0, prior='gauss', prior_scale=None,
                         batch_size=batch_size, n_epochs=n_epochs, optimizer=optimizer,
                         normalize_inputs=normalize_inputs, activation=activation, dropout=dropout,
                         conditions=conditions, verbose=verbose, rng=rng, impl=impl, device=device, rank=rank,
                         world=world, group=group, seed=seed, use_graph=use_graph)
        self.lr = lr

    def __str__(self):
        # the reference class defines no __str__; AAERecommender.train prints the object (aae.py:958)
        return "Autoencoder ({0}, {0}, {1}, {0}, {0}) optimized by {2} with learning rate {3}, batch size {4}".format(
            self.n_hidden, self.n_code, self.optimizer, self.lr, self.batch_size)

    def partial_fit(self, X, y=None, condition_data=None, step=None):
        if y is not None:
            raise ValueError("(Semi-)supervised usage not supported")     # aae.py:321-322 (ValueError here)
        return super().partial_fit(X, y=None, condition_data=condition_data, step=step)

    @property
    def disc(self):
        return None


class AAERecommender(Recommender):
    """Adversarially Regularized Recommender (aae.py:873-977)."""

    def __init__(self, adversarial=True, conditions=None, **kwargs):
        super().__init__()
        self.verbose = kwargs.get('verbose', True)
        self.conditions = conditions
        self.model_params = kwargs
        self.adversarial = adversarial
        self.model = None

    def __str__(self):
        desc = "Adversarial Autoencoder" if self.adversarial else "Autoencoder"
        if self.conditions:
            desc += " conditioned on: " + ', '.join(self.conditions.keys())
        desc += '\nModel Params: ' + str(self.model_params)
        return desc

    def _condition_data(self, bags, fit):
        if not self.conditions:
            return None
        raw = bags.get_attributes(self.conditions.keys())
        return self.conditions.fit_transform(raw) if fit else self.conditions.transform(raw)

    def train(self, training_set):
        print(self)
        X = training_set.tocsr()
        if self.conditions:
            print("Fit transforming conditions:", self.conditions)
        else:
            print("Start of training, not using condition...", self.conditions)
        condition_data = self._condition_data(training_set, fit=True)
        if self.adversarial:
            self.model = AdversarialAutoEncoder(conditions=self.conditions, **self.model_params)
        else:
            self.model = AutoEncoder(conditions=self.conditions, **self.model_params)
        print(self.model)
        print(self.conditions)
        self.model.fit(X, condition_data=condition_data)

    def predict(self, test_set):
        X = test_set.tocsr()
        condition_data = self._condition_data(test_set, fit=False)
        return self.model.predict(X, condition_data=condition_data)

    def predict_topk(self, test_set, k, mask_known=True, items=None, exclude=None):
        X = test_set.tocsr()
        condition_data = self._condition_data(test_set, fit=False)
        return self.model.predict_topk(X, k, condition_data=condition_data, mask_known=mask_known, items=items,
                                       exclude=exclude)

    def evaluate_topk(self, test_set, gold, metrics, items=None, exclude=None):
        """Ranking metrics of the harness (evaluation.py:70-164, 202-240) on the device: ``gold`` is the sparse
        [n, n_items] matrix of held-out items (``Evaluation.y_test``)."""
        X = test_set.tocsr()
        condition_data = self._condition_data(test_set, fit=False)
        return self.model.evaluate_topk(X, gold, metrics, condition_data=condition_data, items=items, exclude=exclude)
