"""``GDRecommender``: Funk-SVD trained one feature at a time
(reference: mfrec/recommendation/gradient_descent.py:30-120, 299-329, 472-503, 506-545, 577-599,
621-648, 769-802, 879-905).

``train`` (= ``feature_training``) calls ``mfrec_b200.lib.gd_estimator``, the drop-in for the
reference's Cython module."""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib import gd_estimator
from mfrec_b200.recommendation.mf import MFRecommender, _fold_ratings, _fold_rows


class GDRecommender(MFRecommender):
    PARAMETERS_INDEX = {'min_epochs': 'min_epochs',
                        'max_epochs': 'max_epochs',
                        'min_improvement': 'min_improvement',
                        'feature_init': 'feature_init',
                        'learning_rate': 'learning_rate',
                        'learning_rate_users': 'learning_rate_users',
                        'learning_rate_items': 'learning_rate_items',
                        'regularization_model': 'K',
                        'regularization_users_bias': 'K2',
                        'regularization_items_bias': 'K3',
                        'nbr_features': 'dimensionality'}
    NATIVE_PREDICTORS = {'predict_rating': 'predict_rating',
                         'predict_rating_with_bias': 'predict_rating_with_bias'}

    def __init__(self, nbr_users=4, nbr_items=6, parameters=False, filename=False):
        MFRecommender.__init__(self, nbr_users, nbr_items, False)
        self.min_epochs = 275
        self.max_epochs = 275
        self.min_improvement = 0.0001
        self.feature_init = 0.1
        self.learning_rate = 0.001
        self.learning_rate_users = 0.001
        self.learning_rate_items = 0.001
        self.K = 0.05
        self.K2 = 0.01
        self.K3 = 0.01
        self.dimensionality = 40
        if parameters:
            self.set_parameters(parameters)
        self.rmse_history = np.zeros(self.max_epochs)

    def __repr__(self):
        return ('Gradient Descent based Recommendation Engine\nNumber of users: %d\n'
                'Number of items: %d\nDimensionality: %d\n'
                % (self.nbr_users, self.nbr_items, self.dimensionality))

    def get_nbr_ratings(self):
        return self.relationship_matrix.tocoo().data.nonzero()[0].shape[0]

    # ---- training (gradient_descent.py:506-545) ------------------------------------------------------
    def feature_training(self, initialize_model=True, handle_bias=False, verbose=False):
        if initialize_model:
            self.svd_v = np.zeros([self.dimensionality, self.nbr_users]) + self.feature_init
            self.svd_u = np.zeros([self.dimensionality, self.nbr_items]) + self.feature_init
        ratings_index, ratings = self.get_ratings(randomize_order=True)
        if handle_bias:
            self.compute_overall_avg()
            self.compute_items_bias_bk()
            self.compute_users_bias_bk()
            gd_estimator.estimator_loop_with_bias(
                self.min_epochs, self.max_epochs, self.min_improvement, self.dimensionality,
                self.feature_init, self.learning_rate, self.learning_rate_users,
                self.learning_rate_items, self.K, self.overall_bias, self.svd_u, self.svd_v,
                ratings_index, ratings, self.items_bias, self.users_bias, self.nbr_users,
                self.nbr_items, int(verbose))
        else:
            gd_estimator.estimator_loop_without_bias(
                self.min_epochs, self.max_epochs, self.min_improvement, self.dimensionality,
                self.feature_init, self.learning_rate, self.K, self.svd_u, self.svd_v,
                ratings_index, ratings, self.nbr_users, self.nbr_items, int(verbose))

    train = feature_training

    def _init_model(self, initialize_model):
        if initialize_model:
            self.svd_v = np.zeros([self.dimensionality, self.nbr_users]) + self.feature_init
            self.svd_u = np.zeros([self.dimensionality, self.nbr_items]) + self.feature_init

    # ---- development variants (gradient_descent.py:299-329, 472-503, 577-599) -------------------------
    def feature_training2(self, initialize_model=True, verbose=False):
        """One `estimator_subloop` call per epoch and a `predictor_subloop` per feature over a dense
        users x items cache, the epoch control in Python (gradient_descent.py:299-329)."""
        rmse, rmse_last = 2.0, 0.0
        self._init_model(initialize_model)
        ratings_cache = np.zeros(self.nbr_users * self.nbr_items, dtype=np.float64)
        ratings_index, ratings = self.get_ratings()
        for f in range(self.dimensionality):
            epoch = 0
            while epoch < self.min_epochs or rmse <= rmse_last - self.min_improvement:
                rmse_last = rmse
                rmse = gd_estimator.estimator_subloop(
                    f, epoch, self.min_improvement, self.dimensionality, self.feature_init,
                    self.learning_rate, self.K, self.svd_u, self.svd_v, ratings_index, ratings,
                    ratings_cache, self.nbr_users, self.nbr_items, int(verbose))
                epoch += 1
            gd_estimator.predictor_subloop(f, epoch, self.dimensionality, self.feature_init, self.svd_u,
                                           self.svd_v, ratings_index, ratings, ratings_cache,
                                           self.nbr_users, self.nbr_items)

    def feature_training_bias(self, initialize_model=True, handle_bias=False, verbose=False):
        """Learned biases: `estimator_loop_with_learned_bias` started from the precomputed bias
        statistics (gradient_descent.py:472-503); `handle_bias` is unused like in the reference."""
        self._init_model(initialize_model)
        ratings_index, ratings = self.get_ratings(randomize_order=True)
        self.compute_overall_avg()
        self.compute_items_bias_bk()
        self.compute_users_bias_bk()
        gd_estimator.estimator_loop_with_learned_bias(
            self.min_epochs, self.max_epochs, self.min_improvement, self.dimensionality, self.feature_init,
            self.learning_rate, self.learning_rate_users, self.learning_rate_items, self.K, self.K2,
            self.overall_bias, self.svd_u, self.svd_v, ratings_index, ratings, self.items_bias,
            self.users_bias, self.nbr_users, self.nbr_items, int(verbose))

    def feature_training_dev(self, initialize_model=True, probe=None, verbose=False):
        """`estimator_loop` with its per-epoch rmse history, which is returned
        (gradient_descent.py:577-599)."""
        rmse = np.zeros(self.max_epochs * self.dimensionality)
        self._init_model(initialize_model)
        # the reference shuffles (consuming the RNG) and then OVERWRITES both arrays with
        # ratings_iterator() order (gradient_descent.py:588-592): it trains on the unshuffled order
        self.get_ratings(randomize_order=True)
        ratings_index, ratings = self.get_ratings()
        gd_estimator.estimator_loop(
            self.min_epochs, self.max_epochs, self.min_improvement, self.dimensionality, self.feature_init,
            self.learning_rate, self.K, self.svd_u, self.svd_v, ratings_index, ratings, 0, rmse,
            self.nbr_users, self.nbr_items, int(verbose))
        return rmse

    # ---- predictors (gradient_descent.py:621-648) ----------------------------------------------------
    def predict_rating(self, item_index, user_index):
        return np.dot(self.svd_u[:, item_index], self.svd_v[:, user_index]) + 1.0

    predict = predict_rating

    def predict_rating_with_bias(self, item_index, user_index):
        s = np.dot(self.svd_u[:, item_index], self.svd_v[:, user_index])
        return s + self.overall_bias + (self.items_bias[item_index] + self.users_bias[user_index])

    def predict_rating_by_label(self, user_label, item_label):
        return MFRecommender.predict_rating_by_label(self, user_label, item_label, 'predict_rating')

    # ---- top-N over all items (gradient_descent.py:769-802) -------------------------------------------
    def find_user_top_match(self, user_index, nbr_recommendations=5):
        self.relationship_matrix_csc = self.relationship_matrix.T.tocsc()
        return self._topn(user_index, self.nbr_items, nbr_recommendations, 'predict_rating')

    # ---- item-item similarity (gradient_descent.py:827-875): feature 0 is skipped, Pearson default
    def similar_items(self, item_index, nbr_recommendations=2, similarity_threshold=False,
                      similarities_output=False, method='pearson'):
        rows = self.svd_u[1:self.dimensionality, :].T
        if method == 'norm_cosine':   # log(1 + cosine of the rows centred by the per-feature means)
            rows = rows - self.svd_u[1:self.dimensionality, :].mean(axis=1)[None, :]
            return self._similar_rows(rows, item_index, nbr_recommendations, similarity_threshold,
                                      similarities_output, 'cosine', transform=lambda c: float(np.log(1.0 + c)),
                                      tag='items_norm_cosine')
        return self._similar_rows(rows, item_index, nbr_recommendations, similarity_threshold,
                                  similarities_output, method, tag='items_gd', skip_first=(method == 'euclidean'))

    # ---- fold-in (gradient_descent.py:879-905) ----------------------------------------------------------
    def _retrain(self, valid_ids, ratings_index, ratings, update_users, update_items, verbose):
        # the reference passes `ratings[valid_ids,:]` (a 2-D index into a 1-D array) and the
        # unfiltered index; the evident intent is the filtered pair
        gd_estimator.estimator_loop_with_bias_dev(
            self.min_epochs, self.max_epochs, self.min_improvement, self.dimensionality,
            self.feature_init, self.learning_rate, self.learning_rate_users,
            self.learning_rate_items, self.K, self.overall_bias, self.svd_u, self.svd_v,
            np.ascontiguousarray(ratings_index[valid_ids, :]), np.ascontiguousarray(ratings[valid_ids]),
            self.items_bias, self.users_bias, self.nbr_users, self.nbr_items, update_users,
            update_items, int(verbose))

    def retrain_user(self, user_index, ratings_index, ratings, verbose=False):
        valid_ids = np.where(ratings_index[:, 0] == user_index)[0]
        self.init_user_features(user_index)
        self._retrain(valid_ids, ratings_index, ratings, 1, 0, verbose)

    def retrain_item(self, item_index, ratings_index, ratings, verbose=False):
        valid_ids = np.where(ratings_index[:, 1] == item_index)[0]
        self.init_item_features(item_index)
        self._retrain(valid_ids, ratings_index, ratings, 0, 1, verbose)

    # ---- batched fold-in (not in the reference): one device call for many rows ----------------------
    # Each leaves the recommender exactly as the loop of the single-row method over the same rows
    # leaves it when gd_estimator.options["schedule"] is "sequential" -- the reference's own order:
    # svd_u, svd_v, the untouched biases, the numpy RNG (the rows' initial features are drawn in list
    # order before the one native call; training draws nothing), what verbose prints and
    # gd_estimator.last_feature_epochs / last_feature_rmse.  The batch always runs that order; under
    # the default stratified schedule the single-row calls order each row's ratings differently and
    # agree with the batch to float tolerance only.  Everything is validated before anything changes
    # or is drawn: rows must be distinct and in range, and every row needs at least one rating (the
    # loop would train the rows before such a row and then raise; the batch raises up front).
    def retrain_users(self, user_indices, ratings_index, ratings, verbose=False):
        """``for u in user_indices: self.retrain_user(u, ratings_index, ratings, verbose)``."""
        rows = _fold_rows(user_indices, self.nbr_users)
        if rows.shape[0]:
            idx, r = _fold_ratings(rows, 0, self.nbr_items, ratings_index, ratings)
            self._fold_in_batch(_native.FOLD_USERS, rows, idx, r, verbose)

    def retrain_items(self, item_indices, ratings_index, ratings, verbose=False):
        """``for i in item_indices: self.retrain_item(i, ratings_index, ratings, verbose)``."""
        rows = _fold_rows(item_indices, self.nbr_items)
        if rows.shape[0]:
            idx, r = _fold_ratings(rows, 1, self.nbr_users, ratings_index, ratings)
            self._fold_in_batch(_native.FOLD_ITEMS, rows, idx, r, verbose)

    def _fold_in_batch(self, side, rows, ratings_index, ratings, verbose):
        col = 0 if side == _native.FOLD_USERS else 1
        rated = np.isin(rows, ratings_index[:, col])
        if not rated.all():
            raise ValueError('%s %d has no ratings to train on' % ('user' if col == 0 else 'item', rows[~rated][0]))
        init = self.init_user_features if side == _native.FOLD_USERS else self.init_item_features
        for row in rows:
            init(row)
        gd_estimator.fold_in(side, self.min_epochs, self.min_improvement, self.dimensionality,
                             self.feature_init, self.learning_rate, self.K, self.overall_bias, self.svd_u,
                             self.svd_v, ratings_index, ratings, self.items_bias, self.users_bias, rows,
                             int(verbose))
        self.invalidate_model()   # a few rows changed in place: the sampled fingerprint may miss them
