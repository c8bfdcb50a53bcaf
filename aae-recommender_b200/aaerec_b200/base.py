"""The recommender plugin contract -- the Python side of the drop-in boundary.

The reference's harness (``Evaluation.__call__``, evaluation.py:355-366) and scripts (main.py:98-124, eval/*.py) talk to
a recommender through two calls only, declared by the ABC of aaerec/base.py:5-19; this module restates that contract for
the B200 classes (and for ``isinstance`` checks of code that imports it from here):

    train(training_set)   training_set: a ``Bags``-like object -- only ``.tocsr()`` (scipy CSR [n, n_items] of ones),
                          ``.get_attributes(keys)`` and ``.size()`` are used (aae.py:942-946)
    predict(test_set)     -> array-like [n, n_items] of scores (the harness masks known items and ranks them,
                          evaluation.py:366-388)

``use_wandb`` is read by the reference's model classes; the B200 classes never log to wandb.  The two ``*_topk``
methods are additions of this package (defaults keep the reference's behaviour): recommenders that can rank on the
device override them.
"""
import abc


class Recommender(abc.ABC):
    use_wandb = False

    @abc.abstractmethod
    def train(self, training_set):
        """Fit the model on the item sets (and attributes) of ``training_set``."""

    @abc.abstractmethod
    def predict(self, test_set):
        """Scores [n, n_items] for the item sets of ``test_set`` (float32; higher = more likely missing)."""

    def predict_topk(self, test_set, k, mask_known=True, items=None, exclude=None):
        """Top-k unknown items per set = argtopk(remove_non_missing(predict(test_set), X), k) without the dense matrix;
        ``items`` / ``exclude`` restrict the candidates (``AdversarialAutoEncoder.predict_topk``)."""
        raise NotImplementedError("%s ranks through predict() only" % type(self).__name__)

    def evaluate_topk(self, test_set, gold, metrics, items=None, exclude=None):
        """The harness' ranking metrics (evaluation.py:70-164, 202-240) computed from device-side ranks; ``items`` /
        ``exclude`` evaluate the candidate-restricted list of ``predict_topk``
        (``AdversarialAutoEncoder.evaluate_topk``)."""
        raise NotImplementedError("%s evaluates through predict() only" % type(self).__name__)
