"""B200-native Denoising Autoencoder behind the reference's API (aaerec/dae.py:144-382; SURVEY 8(f)-3).

The reference's DAE is its plain autoencoder step on a corrupted batch: ``ae_step`` (dae.py:189-210) encodes
``self.corrupt(batch, noise_factor)``, decodes, and takes the BCE against ``batch`` -- and because ``zeros_noise``
(dae.py:48-52) zeroes the entries of ``batch`` IN PLACE, input and target are the same thinned item sets.  Encoder,
Decoder, optimizers (enc_optim / dec_optim at ``lr``), shuffle and batching are those of ``AutoEncoder``.  So the
accelerated DAE is the AutoEncoder engine with one extra kernel in front of every training step
(``aae_batch_corrupt``: drop each CSR entry with probability ``noise_factor``); predict is unchanged.

``corrupt='gauss'`` (dense Gaussian noise on all n_items inputs, dae.py:40-45) makes the input dense and is outside
the accelerated envelope (``NotImplementedError``; no CPU fallback).
"""
import numpy as np
import torch

from .aae import AutoEncoder, _check_conditions, _draw_step_rng, log_losses
from .base import Recommender

NOISE_TYPES = ('gauss', 'zeros')


class DenoisingAutoEncoder(AutoEncoder):
    """dae.py:144-314: same constructor kwargs and defaults."""

    def __init__(self, n_hidden=100, n_code=50, lr=0.001, batch_size=100, n_epochs=500, optimizer='adam',
                 normalize_inputs=True, activation='ReLU', dropout=(.2, .2), noise_factor=0.2, corrupt='zeros',
                 conditions=None, verbose=True, rng='native', impl='auto', device=None, rank=0, world=1, group=None,
                 seed=0, use_graph=True):
        if corrupt.lower() not in NOISE_TYPES:
            raise KeyError(corrupt)                       # NOISE_TYPES[corrupt.lower()] in the reference (dae.py:171)
        if corrupt.lower() != 'zeros':
            raise NotImplementedError("accelerated path supports corrupt='zeros' only: Gaussian noise on every input "
                                      "makes the batch dense")
        super().__init__(n_hidden=n_hidden, n_code=n_code, lr=lr, batch_size=batch_size, n_epochs=n_epochs,
                         optimizer=optimizer, normalize_inputs=normalize_inputs, activation=activation, dropout=dropout,
                         conditions=conditions, verbose=verbose, rng=rng, impl=impl, device=device, rank=rank,
                         world=world, group=group, seed=seed, use_graph=use_graph)
        self.noise_factor = noise_factor
        self.corrupt = corrupt.lower()

    def __str__(self):
        return "Denoising Autoencoder ({0}, {0}, {1}, {0}, {0}) optimized by {2} with learning rate {3}, batch size " \
               "{4}, {5} noise {6}".format(self.n_hidden, self.n_code, self.optimizer, self.lr, self.batch_size,
                                           self.corrupt, self.noise_factor)

    # the reference draws torch.rand(batch.size()) BEFORE the dropout masks of the step (dae.py:191)
    def _corrupt_and_draw(self, B):
        eng = self.engine
        noise = None
        if self.rng == 'oracle':
            noise = torch.rand((B, eng.V))
        eng.corrupt_batch(B, float(self.noise_factor), noise)
        draws = self._draws(B)
        if draws is not None:
            eng.set_rng_draws(B, draws)
        return draws is not None

    def _train_batch_in_buffers(self, B, leaves):
        injected = self._corrupt_and_draw(B)
        self.engine.train_step(B, injected)
        self._cond_end(leaves, B)

    def partial_fit(self, X, y=None, condition_data=None, step=None):
        if y is not None:
            raise ValueError("(Semi-)supervised usage not supported")          # dae.py:216-217
        use_condition = _check_conditions(self.conditions, condition_data)
        if self.engine is None:
            code_size = self.n_code + (self.conditions.size_increment() if use_condition else 0)
            self._build(X.shape[1], code_size)
        indptr, indices = self._csr_batch(X)
        B = int(indptr.shape[0]) - 1
        self.train()
        rows, leaves = self._cond_begin(condition_data if use_condition else None, B)
        self.engine.upload_csr(indptr, indices, rows)
        self._train_batch_in_buffers(B, leaves)
        if self.verbose:
            log_losses(*self.losses())
        return self

    def ae_step(self, batch, condition_data=None):
        raise NotImplementedError("the corruption and the reconstruction step are one call here: use partial_fit")

    def fit(self, X, y=None, condition_data=None):
        """dae.py:232-284 -- AutoEncoder.fit with the corruption kernel in front of every step."""
        self._fit_step = self._train_batch_in_buffers
        try:
            return super().fit(X, y=y, condition_data=condition_data)
        finally:
            self._fit_step = None


class DAERecommender(Recommender):
    """Denoising Recommender (dae.py:317-382): same constructor, ``train`` / ``predict`` on Bags."""

    def __init__(self, conditions=None, **kwargs):
        super().__init__()
        self.verbose = kwargs.get('verbose', True)
        self.model_params = kwargs
        self.conditions = conditions
        self.dae = None

    def __str__(self):
        desc = "Denoising Autoencoder"
        if self.conditions:
            desc += " conditioned on: " + ', '.join(self.conditions.keys())
        desc += '\nDAE Params: ' + str(self.model_params)
        return desc

    def _condition_data(self, bags, fit):
        if not self.conditions:
            return None
        raw = bags.get_attributes(self.conditions.keys())
        return self.conditions.fit_transform(raw) if fit else self.conditions.transform(raw)

    def train(self, training_set):
        X = training_set.tocsr()
        condition_data = self._condition_data(training_set, fit=True)
        self.dae = DenoisingAutoEncoder(conditions=self.conditions, **self.model_params)
        print(self)
        print(self.dae)
        print(self.conditions)
        self.dae.fit(X, condition_data=condition_data)

    def predict(self, test_set):
        X = test_set.tocsr()
        return self.dae.predict(X, condition_data=self._condition_data(test_set, fit=False))

    def predict_topk(self, test_set, k, mask_known=True, items=None, exclude=None):
        X = test_set.tocsr()
        return self.dae.predict_topk(X, k, condition_data=self._condition_data(test_set, fit=False),
                                     mask_known=mask_known, items=items, exclude=exclude)

    def evaluate_topk(self, test_set, gold, metrics, items=None, exclude=None):
        X = test_set.tocsr()
        return self.dae.evaluate_topk(X, gold, metrics, condition_data=self._condition_data(test_set, fit=False),
                                      items=items, exclude=exclude)
