"""Stand-alone stand-ins for the reference's wrapper classes, used only when ``recpack`` itself is not
importable (see ``_ref.py``).  They keep the contract of recpack/algorithms/base.py:33-304 and
recpack/metrics/base.py:21-295 -- ``fit`` / ``predict`` wrappers with input coercion and the two checks,
``name`` / ``identifier``, ``calculate`` -> ``value`` / ``results`` -- in as little code as that takes."""
from __future__ import annotations

import logging
import time
import warnings

import numpy as np
import pandas as pd
from sklearn.base import BaseEstimator
from sklearn.utils.validation import check_is_fitted

logger = logging.getLogger("recpack")


class Algorithm(BaseEstimator):
    @property
    def name(self):
        return type(self).__name__

    @property
    def identifier(self):
        return f"{self.name}({','.join(f'{k}={v}' for k, v in self.get_params().items())})"

    def __str__(self):
        return self.name

    def set_params(self, **params):
        super().set_params(**params)

    def _check_fit_complete(self):
        check_is_fitted(self)

    def fit(self, X):
        t0 = time.time()
        self._fit(self._transform_fit_input(X))
        self._check_fit_complete()
        logger.info(f"Fitting {self.name} complete - Took {time.time() - t0 :.3}s")
        return self

    def predict(self, X):
        self._check_fit_complete()
        X = self._transform_predict_input(X)
        X_pred = self._predict(X)
        self._check_prediction(X_pred, X)
        return X_pred


class ItemSimilarityMatrixAlgorithm(Algorithm):
    pass


class TopKItemSimilarityMatrixAlgorithm(ItemSimilarityMatrixAlgorithm):
    def __init__(self, K):
        super().__init__()
        self.K = K


class FactorizationAlgorithm(Algorithm):
    """Constructor and fit check of recpack/algorithms/base.py:307-369."""

    def __init__(self, num_components=100):
        super().__init__()
        self.num_components = num_components

    def _check_fit_complete(self):
        super()._check_fit_complete()
        assert hasattr(self, "user_embedding_")
        assert hasattr(self, "item_embedding_")


class ItemKNNArgs(TopKItemSimilarityMatrixAlgorithm):
    """Constructor contract of recpack/algorithms/nearest_neighbour.py:170-202."""

    SUPPORTED_SIMILARITIES = ["cosine", "conditional_probability"]

    def __init__(self, K=200, similarity="cosine", pop_discount=None, normalize_X=False, normalize_sim=False):
        super().__init__(K)
        if similarity not in self.SUPPORTED_SIMILARITIES:
            raise ValueError(f"similarity {similarity} not supported")
        if similarity != "conditional_probability" and pop_discount:
            warnings.warn("pop_discount only applies to conditional probability similarity; it is ignored here.", UserWarning)
        if type(pop_discount) == float and not 0 <= pop_discount <= 1:
            raise ValueError("Invalid value for pop_discount. Value should be between 0 and 1.")
        self.similarity, self.pop_discount = similarity, pop_discount
        self.normalize_X, self.normalize_sim = normalize_X, normalize_sim


class MetricTopK:
    def __init__(self, K):
        self.num_users_ = 0
        self.num_items_ = 0
        self.K = K

    @property
    def name(self):
        return f"{type(self).__name__}_{self.K}"

    @property
    def num_items(self):
        return self.num_items_

    @property
    def num_users(self):
        return self.num_users_

    @property
    def value(self):
        return self.value_

    def _verify_shape(self, y_true, y_pred):
        if y_true.shape != y_pred.shape:
            raise AssertionError(f"Shape mismatch between y_true: {y_true.shape} and y_pred: {y_pred.shape}")
        return True

    def _map_users(self, users):
        return self.user_id_map_[users] if hasattr(self, "user_id_map_") else users


class ListwiseMetricK(MetricTopK):
    col_names = ["user_id", "score"]

    @property
    def results(self):
        scores = self.scores_.toarray().ravel()
        return pd.DataFrame(dict(zip(self.col_names, (self._map_users(np.arange(len(scores))), scores))))

    @property
    def value(self):
        return self.scores_.mean()


class ElementwiseMetricK(MetricTopK):
    col_names = ["user_id", "item_id", "score"]

    @property
    def results(self):
        scores = self.scores_.toarray()
        int_users, items = self.y_pred_top_K_.nonzero()
        values = scores[int_users, items]
        missing = sorted(set(range(scores.shape[0])) - set(int_users.tolist()))
        if missing:  # users without recommendations: K rows with item_id = NaN and score 0
            int_users = np.concatenate([int_users, np.repeat(missing, self.K)])
            items = np.concatenate([items.astype(float), np.full(len(missing) * self.K, np.nan)])
            values = np.concatenate([values, np.zeros(len(missing) * self.K)])
        return pd.DataFrame(dict(zip(self.col_names, (self._map_users(int_users), items, values))))

    @property
    def value(self):
        return self.scores_.sum(axis=1).mean()


class GlobalMetricK(MetricTopK):
    @property
    def results(self):
        return pd.DataFrame({"score": [self.value]})
