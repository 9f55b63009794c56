"""``KMFRecommender``: kernel matrix factorisation trained by SGD
(reference: mfrec/recommendation/kmf.py; Rendle & Schmidt-Thieme, RecSys 2008).

``train`` hands the reference's own arrays to ``mfrec_b200.lib.kmf_train`` -- the drop-in for the
Cython module the reference imports (kmf.py:18, with its broken package path fixed)."""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib import kmf_train
from mfrec_b200.recommendation.base import Error
from mfrec_b200.recommendation.mf import MFRecommender, _fold_ratings, _fold_rows

_KERNELS = {'train_logistic_kernel': kmf_train.train_logistic_kernel,
            'train_linear_kernel': kmf_train.train_linear_kernel}
_KERNEL_IDS = {'train_logistic_kernel': _native.KERNEL_LOGISTIC,
               'train_linear_kernel': _native.KERNEL_LINEAR}


def _fold_in(kernel, *args):
    """A fold-in trains a handful of ratings against a frozen side: run it in the reference's own
    order and precision (sequential schedule: float64, bit-exact for the linear kernel).  The library
    then moves only the rows the ratings name, so the frozen factors stay bit-identical like in
    the reference (a stratified fp32 pass would round every row of the model in place)."""
    saved = kmf_train.options["schedule"]
    kmf_train.options["schedule"] = "sequential"
    try:
        return _KERNELS[kernel](*args)
    finally:
        kmf_train.options["schedule"] = saved


class KMFRecommender(MFRecommender):
    # As in the reference (kmf.py:33-42) the three regularisation keys map to K / K2 / K3 while
    # training reads K_users / K_items / K_bias: those settings are silently ignored there, and
    # here.  Set the attributes directly to change them.
    PARAMETERS_INDEX = {'nbr_epochs': 'nbr_epochs',
                        'min_improvement': 'min_improvement',
                        'feature_init': 'feature_init',
                        'learning_rate': 'learning_rate',
                        'learning_rate_users': 'learning_rate_users',
                        'learning_rate_items': 'learning_rate_items',
                        'regularization_users': 'K',
                        'regularization_items': 'K2',
                        'regularization_bias': 'K3',
                        'nbr_features': 'dimensionality'}
    NATIVE_PREDICTORS = {'predict_logistic': 'predict_logistic', 'predict_linear': 'predict_linear',
                         'predict_linear_neg': 'predict_linear_neg'}

    def __init__(self, nbr_users=4, nbr_items=6, parameters=False, filename=False):
        MFRecommender.__init__(self, nbr_users, nbr_items, False)
        self.nbr_epochs = 200
        self.feature_init = 0.1
        self.learning_rate = 0.01
        self.learning_rate_users = 0.01
        self.learning_rate_items = 0.01
        self.K_users = 0.1
        self.K_items = 0.1
        self.K_bias = 0.007
        self.dimensionality = 40
        if parameters:
            self.set_parameters(parameters)

    def __repr__(self):
        return ('Kernel Matrix Factorization Recommendation Engine\n'
                'Number of users: %d\nNumber of items: %d\n' % (self.nbr_users, self.nbr_items))

    # ---- predictors (kmf.py:79-103): (item_index, user_index) ------------------------------------
    def _raw(self, item_index, user_index):
        s = np.dot(self.svd_u[:, item_index], self.svd_v[:, user_index])
        return s + (self.items_bias[item_index] + self.users_bias[user_index])

    def predict_logistic(self, item_index, user_index):
        s = self._raw(item_index, user_index)
        return self.min_rating + (1.0 / (1.0 + np.exp(-s))) * (self.max_rating - self.min_rating)

    def predict_linear(self, item_index, user_index):
        return self._raw(item_index, user_index)

    def predict_linear_neg(self, item_index, user_index):
        return self.min_rating + self._raw(item_index, user_index) * (self.max_rating - self.min_rating)

    predict = predict_logistic

    # ---- training (kmf.py:197-220) -------------------------------------------------------------------
    def train(self, initialize_model=True, verbose=False, kernel='train_logistic_kernel'):
        self.relationship_matrix_csc = self.relationship_matrix.T.tocsc()
        if initialize_model:
            self.init_feature_normal(0.0, 0.1)
        ratings_index, ratings = self.get_ratings(randomize_order=True)
        self.compute_overall_avg()
        self.items_bias = np.zeros(self.nbr_items)
        self.users_bias = np.zeros(self.nbr_users)
        _KERNELS[kernel](self.nbr_epochs, self.dimensionality, self.feature_init, self.learning_rate,
                         self.learning_rate_users, self.learning_rate_items, self.K_users,
                         self.K_items, self.K_bias, self.overall_bias, self.svd_u, self.svd_v,
                         ratings_index, ratings, self.items_bias, self.users_bias, 1, 1, int(verbose))

    # ---- fold-in (kmf.py:120-146) --------------------------------------------------------------------
    def retrain_user(self, user_index, ratings_index, ratings, verbose=False, kernel='train_logistic_kernel'):
        valid_ids = np.where(ratings_index[:, 0] == user_index)[0]
        self.init_user_features(user_index)
        _fold_in(kernel, self.nbr_epochs, self.dimensionality, self.feature_init, self.learning_rate,
                         self.learning_rate_users, self.learning_rate_items, self.K_users,
                         self.K_items, self.K_bias, self.overall_bias, self.svd_u, self.svd_v,
                         np.ascontiguousarray(ratings_index[valid_ids, :]),
                         np.ascontiguousarray(ratings[valid_ids]), self.items_bias, self.users_bias,
                         1, 0, int(verbose))

    def retrain_item(self, item_index, ratings_index, ratings, verbose=False, kernel='train_logistic_kernel'):
        # the reference's call (kmf.py:144-146) drops the ratings_index argument and cannot run;
        # this is the evident intent, symmetric to retrain_user
        valid_ids = np.where(ratings_index[:, 1] == item_index)[0]
        self.init_item_features(item_index)
        _fold_in(kernel, self.nbr_epochs, self.dimensionality, self.feature_init, self.learning_rate,
                         self.learning_rate_users, self.learning_rate_items, self.K_users,
                         self.K_items, self.K_bias, self.overall_bias, self.svd_u, self.svd_v,
                         np.ascontiguousarray(ratings_index[valid_ids, :]),
                         np.ascontiguousarray(ratings[valid_ids]), self.items_bias, self.users_bias,
                         0, 1, int(verbose))

    def add_user(self, user_label, users_ratings_index, users_ratings):
        """Fold a new user in without touching the relationship matrix (kmf.py:149-172)."""
        if users_ratings_index.shape[0] != users_ratings.shape[0]:
            raise Error('The index and the ratings array must be the same size')
        new_id = self._get_new_user_id()
        self.users_index[user_label] = new_id
        self.users_label[new_id] = user_label
        self.svd_v = np.ascontiguousarray(np.c_[self.svd_v, np.zeros(self.dimensionality)])
        self.users_bias = np.r_[self.users_bias, 0.0]
        ratings_index = np.zeros([users_ratings.shape[0], 2], dtype=np.int32)
        ratings_index[:, 0] = new_id
        ratings_index[:, 1] = users_ratings_index
        self.retrain_user(new_id, ratings_index, np.asarray(users_ratings, dtype=np.float64))
        return new_id

    # ---- batched fold-in (not in the reference): one device call for many rows ----------------------
    # Each leaves the recommender exactly as the loop of the single-row method over the same rows
    # would: factors, biases, index / label maps and the numpy RNG (the new rows' initial features
    # are drawn in list order before the one native call; training draws nothing).  Everything is
    # validated before anything changes or is drawn.  Rows must be distinct and in range.
    def retrain_users(self, user_indices, ratings_index, ratings, verbose=False, kernel='train_logistic_kernel'):
        """``for u in user_indices: self.retrain_user(u, ratings_index, ratings, verbose, kernel)``."""
        kernel_id = _KERNEL_IDS[kernel]
        rows = _fold_rows(user_indices, self.nbr_users)
        if rows.shape[0]:
            idx, r = _fold_ratings(rows, 0, self.nbr_items, ratings_index, ratings)
            self._fold_in_batch(_native.FOLD_USERS, rows, idx, r, verbose, kernel_id)

    def retrain_items(self, item_indices, ratings_index, ratings, verbose=False, kernel='train_logistic_kernel'):
        """``for i in item_indices: self.retrain_item(i, ratings_index, ratings, verbose, kernel)``."""
        kernel_id = _KERNEL_IDS[kernel]
        rows = _fold_rows(item_indices, self.nbr_items)
        if rows.shape[0]:
            idx, r = _fold_ratings(rows, 1, self.nbr_users, ratings_index, ratings)
            self._fold_in_batch(_native.FOLD_ITEMS, rows, idx, r, verbose, kernel_id)

    def add_users(self, user_labels, users_ratings_index_list, users_ratings_list, verbose=False,
                  kernel='train_logistic_kernel'):
        """``[self.add_user(l, i, r) for l, i, r in zip(...)]`` (add_user trains with the logistic
        kernel, silently; ``kernel`` / ``verbose`` choose otherwise).  Returns the new user ids."""
        kernel_id = _KERNEL_IDS[kernel]
        labels, items_list, ratings_list = list(user_labels), list(users_ratings_index_list), list(users_ratings_list)
        if not len(labels) == len(items_list) == len(ratings_list):
            raise ValueError('user_labels, users_ratings_index_list and users_ratings_list differ in length')
        first, n = self.nbr_users, len(labels)
        if n == 0:
            return []
        idx, r = [], []
        for j, (items, ratings) in enumerate(zip(items_list, ratings_list)):
            items, ratings = np.asarray(items), np.asarray(ratings, dtype=np.float64)
            if items.shape[0] != ratings.shape[0]:
                raise Error('The index and the ratings array must be the same size')
            ratings_index = np.zeros([ratings.shape[0], 2], dtype=np.int32)
            ratings_index[:, 0] = first + j
            ratings_index[:, 1] = items
            idx.append(ratings_index)
            r.append(ratings)
        rows = np.arange(first, first + n)
        idx, r = _fold_ratings(rows, 0, self.nbr_items, np.concatenate(idx), np.concatenate(r))
        for label in labels:
            new_id = self._get_new_user_id()
            self.users_index[label] = new_id
            self.users_label[new_id] = label
        self.svd_v = np.ascontiguousarray(np.c_[self.svd_v, np.zeros((self.dimensionality, n))])
        self.users_bias = np.r_[self.users_bias, np.zeros(n)]
        self._fold_in_batch(_native.FOLD_USERS, rows, idx, r, verbose, kernel_id)
        return [int(x) for x in rows]

    def _fold_in_batch(self, side, rows, ratings_index, ratings, verbose, kernel_id):
        init = self.init_user_features if side == _native.FOLD_USERS else self.init_item_features
        for row in rows:
            init(row)
        kmf_train.fold_in(kernel_id, side, self.nbr_epochs, self.dimensionality, self.learning_rate,
                          self.K_users, self.K_items, self.K_bias, self.svd_u, self.svd_v, ratings_index,
                          ratings, self.items_bias, self.users_bias, rows, int(verbose))
        self.invalidate_model()   # a few rows changed in place: the sampled fingerprint may miss them

