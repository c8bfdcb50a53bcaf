"""B200-native DecodingRecommender behind the reference's API (aaerec/aae.py:461-584; SURVEY 8(f)-3).

"Only the decoder part of the AAE, basically 2-MLP": the reference's ``Decoder`` (aae.py:149-178) maps the
concatenated condition encodings of a record (aae.py:495-507: the first encoded condition, every further one imposed
= concatenated on it) to sigmoid scores over all items, trained with ``F.binary_cross_entropy(y_pred + TINY,
y + TINY)`` and one Adam at ``lr`` (aae.py:508-513, 522-523).  Here: ``aae_decoder_fwd`` -> the fused output-layer
kernel K3 (``aae_dec_out_train_ws``: lin3 + sigmoid + BCE + backward + Adam in one pass over lin3) ->
``aae_decoder_bwd`` -> ``aae_decoder_wgrad``; predict = ``aae_decoder_fwd`` (eval) + the dense scores kernel, or the
fused top-k tail (``predict_topk``).  Shuffle, batching and the condition plumbing are those of the AutoEncoder
classes (device-side epoch feed; trainable conditions through their Python protocol with the kernels' gradient).
"""
import torch

from .aae import AutoEncoder, _ModuleView
from .base import Recommender
from .engine_siblings import DecoderEngine


def _init_decoder_params(code_size, n_hidden, n_items):
    """``Decoder(code_size, n_hidden, n_items)`` (aae.py:152-155): lin1, lin2, lin3 in construction order, stock
    nn.Linear init on the CPU generator."""
    out = {}
    for name, fin, fout in (("lin1", code_size, n_hidden), ("lin2", n_hidden, n_hidden), ("lin3", n_hidden, n_items)):
        lin = torch.nn.Linear(fin, fout)
        out[name + ".weight"] = lin.weight.detach()
        out[name + ".bias"] = lin.bias.detach()
    return out


class _DecoderNet(AutoEncoder):
    """The model object behind DecodingRecommender: AutoEncoder's fit / partial_fit / predict / predict_topk loops on a
    ``DecoderEngine`` (no encoder, code = the condition rows)."""
    _announce = False

    def __init__(self, n_hidden=100, lr=0.001, batch_size=100, n_epochs=100, optimizer='adam', activation='ReLU',
                 dropout=(.2, .2), conditions=None, verbose=True, **kw):
        super().__init__(n_hidden=n_hidden, n_code=0, lr=lr, batch_size=batch_size, n_epochs=n_epochs,
                         optimizer=optimizer, activation=activation, dropout=dropout, conditions=conditions,
                         verbose=verbose, **kw)

    def __str__(self):
        return "MLP-2 Decoder ({0}, {0}) optimized by {1} with learning rate {2}".format(self.n_hidden, self.optimizer,
                                                                                       self.lr)

    def _build(self, n_items, code_size, params=None):
        if self.world != 1:
            raise NotImplementedError("DecodingRecommender runs on one GPU")
        if params is None:
            params = _init_decoder_params(code_size, self.n_hidden, n_items)
        self.engine = DecoderEngine(n_items, self.n_hidden, cond_dim=code_size, lr=self.lr, dropout=self.dropout,
                                    device=self.device, impl=self.impl, seed=self.seed, max_batch=self.batch_size,
                                    use_graph=self.use_graph)
        self.engine.load_params(params)
        self.last_losses = None

    def _draws(self, B):
        """Decoder.forward draws drop1 then drop2 (aae.py:165-175) -- nothing else in a step."""
        if self.rng != 'oracle':
            return None
        p1, p2 = self.dropout

        def mask(p):
            if p == 0:
                return None
            return torch.empty((B, self.n_hidden), dtype=torch.float32).bernoulli_(1 - p).div_(1 - p)
        return {"ae_dec": (mask(p1), mask(p2))}

    def _log_losses(self, losses):
        print("\rLoss: {}".format(losses[0]), flush=True, end='')          # aae.py:517-518

    enc = dec = disc = None

    @property
    def mlp(self):
        if self.engine is None:
            return None
        return _ModuleView({"mlp." + k: v for k, v in self.engine.state_dict().items()}, "mlp")


class DecodingRecommender(Recommender):
    """ Only the decoder part of the AAE, basically 2-MLP (aae.py:461-584): same constructor, ``train`` / ``predict``
    on Bags, ``fit(condition_data, Y)`` / ``partial_fit(condition_data, y)``. """

    def __init__(self, conditions, n_epochs=100, batch_size=100, optimizer='adam', n_hidden=100, lr=0.001, verbose=True,
                 **mlp_params):
        super().__init__()
        self.n_epochs = n_epochs
        self.batch_size = batch_size
        self.lr = lr
        self.optimizer = optimizer.lower()
        self.model_params = mlp_params
        self.verbose = verbose
        self.n_hidden = n_hidden
        assert len(conditions), "Minimum 1 condition is necessary for MLP"
        self.conditions = conditions
        self.model = None
        self.mlp_optim, self.vect = None, None

    def __str__(self):
        desc = "MLP-2 Decoder with " + str(self.n_hidden) + " hidden units"
        desc += " training for " + str(self.n_epochs)
        desc += " optimized by " + self.optimizer
        desc += " with learning rate " + str(self.lr)
        desc += " with %d conditions: %s " % (len(self.conditions), ', '.join(self.conditions.keys()))
        desc += "\n MLP Params: " + str(self.model_params)
        return desc

    @property
    def mlp(self):
        return self.model.mlp if self.model is not None else None

    def _make_model(self):
        # mlp_params are the Decoder's keyword arguments (aae.py:150-151: dropout, activation) plus this package's
        # engine options (rng, impl, device, seed, use_graph)
        self.model = _DecoderNet(n_hidden=self.n_hidden, lr=self.lr, batch_size=self.batch_size, n_epochs=self.n_epochs,
                                 optimizer=self.optimizer, conditions=self.conditions, verbose=self.verbose,
                                 **self.model_params)
        self.mlp_optim = self.model.dec_optim

    def partial_fit(self, condition_data, y, step=None):
        """aae.py:490-520 (``y``: the batch's item sets, dense tensor / ndarray as the reference passes, or sparse)."""
        if self.model is None:
            self._make_model()
        if torch.is_tensor(y):
            y = y.detach().cpu().numpy()
        self.model.partial_fit(y, condition_data=condition_data)
        return self

    def fit(self, condition_data, Y):
        """aae.py:522-545."""
        self._make_model()
        self.model.fit(Y, condition_data=condition_data)
        return self

    def train(self, training_set):
        Y = training_set.tocsr()
        condition_data_raw = training_set.get_attributes(self.conditions.keys())
        condition_data = self.conditions.fit_transform(condition_data_raw)
        self.fit(condition_data, Y)

    def _query(self, test_set):
        condition_data_raw = test_set.get_attributes(self.conditions.keys())
        return test_set.tocsr(), self.conditions.transform(condition_data_raw)

    def predict(self, test_set):
        """aae.py:555-584: float32 [n, n_items] sigmoid scores from the conditions alone."""
        X, condition_data = self._query(test_set)
        return self.model.predict(X, condition_data=condition_data)

    def predict_topk(self, test_set, k, mask_known=True, items=None, exclude=None):
        X, condition_data = self._query(test_set)
        return self.model.predict_topk(X, k, condition_data=condition_data, mask_known=mask_known, items=items,
                                       exclude=exclude)

    def evaluate_topk(self, test_set, gold, metrics, items=None, exclude=None):
        X, condition_data = self._query(test_set)
        return self.model.evaluate_topk(X, gold, metrics, condition_data=condition_data, items=items, exclude=exclude)
