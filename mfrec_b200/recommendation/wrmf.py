"""``WRMFRecommender``: weighted regularised matrix factorisation for implicit feedback, trained by
alternating least squares (reference: mfrec/recommendation/wrmf.py; Hu, Koren, Volinsky, ICDM 2008).
The reference's only runnable example (examples/example1b_movielens_100k_wrmf.py) uses this class
with ``metrics.precision_recall``."""
import numpy as np

from mfrec_b200.lib.als_implicit import als_wrmf
from mfrec_b200.lib.datasets import create_bool_sparse_col, create_bool_sparse_row
from mfrec_b200.recommendation.mf import MFRecommender


class WRMFRecommender(MFRecommender):
    PARAMETERS_INDEX = {'nbr_epochs': 'nbr_epochs',
                        'feature_init': 'feature_init',
                        'regularization_model': 'K',
                        'neighborhood': 'neighborhood',
                        'nbr_features': 'dimensionality'}
    NATIVE_PREDICTORS = {'predict': 'predict_dot'}

    def __init__(self, nbr_users=4, nbr_items=6, parameters=None):
        MFRecommender.__init__(self, nbr_users, nbr_items, False)
        self.nbr_epochs = 20
        self.feature_init = 0.1
        self.K = 0.025
        self.dimensionality = 20
        self.neighborhood = 500
        if parameters:
            self.set_parameters(parameters)

    def __repr__(self):
        return ('Weighted Regularized Matrix Factorization Recommendation Engine\n'
                'Number of users: %d\nNumber of items: %d\n' % (self.nbr_users, self.nbr_items))

    def predict(self, item_index, user_index):
        return np.dot(self.svd_u[:, item_index], self.svd_v[:, user_index])

    def predict_rating_by_label(self, user_label, item_label):
        try:
            return self.predict(self.items_index[item_label], self.users_index[user_label])
        except KeyError:
            return 0.0

    def train(self, initialize_model=True, handle_bias=False, verbose=False):
        """wrmf.py:83-110.  As in the reference the regularisation handed to the kernel is the
        literal 0.015 and c_pos the literal 1 (the ``K`` attribute is not used there either).
        Note (a property of the reference, kept): the constant initialisation makes all features
        identical; round-off breaks the symmetry and from the third epoch on the factors depend on
        the linear solver's rounding (tests/test_als_gpu.py).  With several devices in
        ``mfrec_b200.lib.als_implicit.options["devices"]`` the rows of each half-pass are split over
        them; the factors are the same bit for bit as on the first of them alone."""
        self.relationship_matrix_csc = self.relationship_matrix.T.tocsc()
        if initialize_model:
            self.svd_v = np.zeros([self.dimensionality, self.nbr_users]) + self.feature_init
            self.svd_u = np.zeros([self.dimensionality, self.nbr_items]) + self.feature_init
        m = np.zeros([self.dimensionality, self.dimensionality])
        m_inv = np.zeros([self.dimensionality, self.dimensionality])
        users_row, users_col = create_bool_sparse_row(self.relationship_matrix)
        items_row, items_col = create_bool_sparse_col(self.relationship_matrix)
        self.compute_overall_avg()
        als_wrmf(self.nbr_epochs, self.dimensionality, self.svd_u, self.svd_v, m, m_inv, users_row, users_col,
                 items_row, items_col, self.nbr_users, self.nbr_items, c_pos=1, k=0.015, verbose=verbose)
