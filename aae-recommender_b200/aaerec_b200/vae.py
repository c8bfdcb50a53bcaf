"""B200-native Variational Autoencoder recommender behind the reference's API (aaerec/vae.py:47-340; SURVEY 8(f)-3).

The reference's VAE: ``h1 = relu(fc1(normalize(x)))``, ``mu, logvar = fc21(h1), fc22(h1)``, ``z = eps * exp(logvar/2) +
mu`` (vae.py:103-110), conditions concatenated on ``z`` (vae.py:120-123), ``recon = sigmoid(fc4(relu(fc3(z))))``;
``loss = BCELoss()(recon, x) + KLD`` with ``KLD = -0.5 * sum(1 + logvar - mu^2 - exp(logvar))`` (vae.py:126-145; the
``size_average = False`` assignment after construction has no effect on torch >= 1.0, so the BCE term is the MEAN over
batch x items); ONE Adam at ``lr`` over all parameters (vae.py:90-91); no dropout.

Here: ``fc1`` is the sparse first layer (the W1t row gather of the AAE encoder, with its time-blocked dense-Adam sweep),
``aae_vae_fwd`` / ``aae_vae_bwd`` / ``aae_vae_wgrad`` run the small layers (``csrc/siblings.cu``), and ``fc4`` + sigmoid
+ BCE + backward + Adam is the fused output-layer kernel K3; predict reuses the scores / fused top-k kernels (K5).
The BCE of the reference has no ``+ 1e-12`` here (vae.py:130 vs aae.py:693); the difference (<= 1e-10 per term) is far
below fp32 resolution of the loss, so K3 serves both.

``rng='oracle'``: eps is drawn by ``torch.randn`` on the CPU generator where the reference draws it (one ``[B, n_code]``
draw per forward, also in ``predict`` -- the reference samples in eval mode too, vae.py:252-256) and injected;
``rng='native'``: in-kernel Philox.
"""
import numpy as np
import torch

from .aae import AutoEncoder, _check_conditions, _canonical_csr
from .base import Recommender
from .engine_siblings import VAEEngine

STATUS_FORMAT = "[ R: {:.4f}]"      # vae.py:40


def log_losses(loss):
    print('\r' + STATUS_FORMAT.format(loss), end='', flush=True)


def _init_vae_params(inp, out, n_hidden, n_code, code_size):
    """vae.py:76-87: fc1, fc21, fc22, fc3, fc4 in construction order, stock nn.Linear init on the CPU generator."""
    p = {}
    for name, fin, fout in (("fc1", inp, n_hidden), ("fc21", n_hidden, n_code), ("fc22", n_hidden, n_code),
                            ("fc3", code_size, n_hidden), ("fc4", n_hidden, out)):
        lin = torch.nn.Linear(fin, fout)
        p[name + ".weight"] = lin.weight.detach()
        p[name + ".bias"] = lin.bias.detach()
    return p


class VAE(AutoEncoder):
    """vae.py:47-266: same constructor arguments and defaults (``inp`` / ``out`` = n_items)."""
    _announce = False

    def __init__(self, inp, out, n_hidden=100, n_code=50, lr=0.001, batch_size=100, n_epochs=500, optimizer='adam',
                 normalize_inputs=True, activation='ReLU', final_activation='Sigmoid', conditions=None, verbose=True,
                 log_interval=1, device=None, rng='native', impl='auto', seed=0, use_graph=True, params=None):
        if final_activation != 'Sigmoid':
            raise NotImplementedError("accelerated path supports final_activation='Sigmoid' only (the fused BCE)")
        if inp != out:
            raise NotImplementedError("accelerated path reconstructs its own input: inp == out == n_items")
        super().__init__(n_hidden=n_hidden, n_code=n_code, lr=lr, batch_size=batch_size, n_epochs=n_epochs,
                         optimizer=optimizer, normalize_inputs=normalize_inputs, activation=activation,
                         dropout=(0.0, 0.0), conditions=conditions, verbose=verbose, rng=rng, impl=impl, device=device,
                         seed=seed, use_graph=use_graph)
        self.inp = inp
        self.log_interval = log_interval
        code_size = n_code + (conditions.size_increment() if conditions else 0)
        if params is None:
            params = _init_vae_params(inp, out, n_hidden, n_code, code_size)
        self.engine = VAEEngine(inp, n_hidden, n_code, cond_dim=code_size - n_code, lr=lr,
                                normalize_inputs=normalize_inputs, device=device, impl=impl, seed=seed,
                                max_batch=batch_size, use_graph=use_graph)
        self.engine.load_params(params)

    def __str__(self):
        return "VAE (fc1 {0}->{1}, fc21/fc22 {1}->{2}, fc3 {3}->{1}, fc4 {1}->{0}) optimized by {4} with learning rate " \
               "{5}, batch size {6}".format(self.inp, self.n_hidden, self.n_code, self.engine.Cp, self.optimizer,
                                            self.lr, self.batch_size)

    def cuda(self):
        return self                       # VAERecommender.train calls self.model.cuda() (vae.py:327-328)

    def _build(self, n_items, code_size, params=None):
        """The reference builds the network in the constructor (vae.py:76-91); fit / partial_fit only check shapes."""
        assert n_items == self.inp and code_size == self.engine.Cp, (n_items, self.inp, code_size, self.engine.Cp)
        if params is not None:
            self.engine.load_params(params)

    def _draws(self, B):
        if self.rng != 'oracle':
            return None
        self.engine.set_eps(B, torch.randn((B, self.n_code), dtype=torch.float32))       # vae.py:109
        return {}                                                                         # no dropout masks

    def losses(self):
        """(BCE mean + KLD, BCE mean, KLD) of the last step (vae.py:145): a device->host read."""
        bce, kld_per_row, _ = (float(x) for x in self.engine.losses.cpu().tolist())
        B = self.engine.last_B
        self.last_losses = (bce + kld_per_row * B, bce, kld_per_row * B)
        return self.last_losses

    def _log_losses(self, losses):
        log_losses(losses[0] / max(self.engine.last_B, 1))          # vae.py:184-185: loss.item() / len(X)

    def partial_fit(self, X, y=None, condition_data=None, step=None):
        if y is not None:
            raise ValueError("(Semi-)supervised usage not supported")                     # vae.py:159-160
        return super().partial_fit(X, y=None, condition_data=condition_data, step=step)

    def predict(self, X, condition_data=None):
        """vae.py:231-266: float32 [n, n_items]; every batch runs the full forward, sampling included (the test-loss
        print of the reference is not reproduced)."""
        eng = self.engine
        eng.eval_injected = self.rng == 'oracle'
        n = X.shape[0]
        out = np.empty((n, eng.V), dtype=np.float32)
        dev = torch.empty(self.batch_size, eng.Vloc, dtype=torch.float32, device=eng.dev)
        for start, end, B in self._iter_batches(X, condition_data):
            if eng.eval_injected:
                eng.set_eps(B, torch.randn((B, self.n_code), dtype=torch.float32))
            eng.scores(B, dev, apply_sigmoid=True)
            out[start:end] = dev[:B].cpu().numpy()
        return out

    def predict_topk(self, X, k, condition_data=None, mask_known=True, return_scores=False, shard="items",
                     items=None, exclude=None):
        self.engine.eval_injected = False          # ranking batches differ from the reference's: native noise
        return super().predict_topk(X, k, condition_data=condition_data, mask_known=mask_known,
                                    return_scores=return_scores, shard=shard, items=items, exclude=exclude)

    def _gold_ranks(self, X, Y, condition_data, batch_size, filt):
        # gold_ranks and evaluate_topk: native noise, as in predict_topk (an oracle-RNG predict leaves its noise set)
        self.engine.eval_injected = False
        return super()._gold_ranks(X, Y, condition_data, batch_size, filt)


class VAERecommender(Recommender):
    """Varietional Autoencoder Recommender (vae.py:269-340): same constructor, ``train`` / ``predict`` on Bags."""

    def __init__(self, conditions=None, **kwargs):
        super().__init__()
        self.verbose = kwargs.get('verbose', True)
        self.conditions = conditions
        self.model_params = kwargs
        self.model = None

    def __str__(self):
        desc = "Variational Autoencoder"
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
        X = training_set.tocsr()
        condition_data = self._condition_data(training_set, fit=True)
        self.model = VAE(X.shape[1], X.shape[1], conditions=self.conditions, **self.model_params)
        print(self)
        print(self.model)
        print(self.conditions)
        self.model.fit(X, condition_data=condition_data)

    def predict(self, test_set):
        X = test_set.tocsr()
        return self.model.predict(X, condition_data=self._condition_data(test_set, fit=False))

    def predict_topk(self, test_set, k, mask_known=True, items=None, exclude=None):
        X = test_set.tocsr()
        return self.model.predict_topk(X, k, condition_data=self._condition_data(test_set, fit=False),
                                       mask_known=mask_known, items=items, exclude=exclude)

    def evaluate_topk(self, test_set, gold, metrics, items=None, exclude=None):
        X = test_set.tocsr()
        return self.model.evaluate_topk(X, gold, metrics, condition_data=self._condition_data(test_set, fit=False),
                                        items=items, exclude=exclude)
