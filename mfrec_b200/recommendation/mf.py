"""``MFRecommender``: shared pieces of the factor-model recommenders
(reference: mfrec/recommendation/mf.py:33-194)."""
import numpy as np

from mfrec_b200 import _native
from mfrec_b200.lib._buffers import buffer_arg, options
from mfrec_b200.recommendation.base import BaseRecommender


class MFRecommender(BaseRecommender):
    # predictor method name -> predictor of the C ABI (include/mfrec_b200.h MFREC_PRED_*)
    NATIVE_PREDICTORS = {}

    def __init__(self, nbr_users=4, nbr_items=6, parameters=False):
        BaseRecommender.__init__(self, nbr_users, nbr_items, parameters)
        self.neighborhood = 500

    def clamping(self, value, min=1.0, max=5.0):
        # the bounds are hard-coded in the reference too (mf.py:44-53)
        if value > 5.0:
            value = 5.0
        if value < 1.0:
            value = 1.0
        return value

    def warmyup(self):
        self.relationship_matrix_csc = self.relationship_matrix.tocsc()

    def predict_rating_by_label(self, user_label, item_label, predictor='predict_logistic'):
        try:
            item_index = self.items_index[item_label]
            user_index = self.users_index[user_label]
            return getattr(self, predictor)(item_index, user_index)
        except KeyError:
            return self.overall_avg

    # ---- BellKor bias statistics (mf.py:78-121): one device pass instead of per-row scipy slicing
    def _bias_stats(self):
        idx, r = self.get_ratings(randomize_order=False)
        mu, ib, ub = _native.bias_stats(idx, r, self.nbr_items, self.nbr_users,
                                        getattr(self, 'K2', 0.01), getattr(self, 'K3', 0.01))
        return mu, ib, ub

    def compute_items_bias_bk(self):
        if not self.overall_bias:
            self.compute_overall_avg()
        _, self.items_bias, _ = self._bias_stats()
        self.relationship_matrix_csc = self.relationship_matrix.tocsc()

    def compute_users_bias_bk(self):
        if not self.overall_bias:
            self.compute_overall_avg()
        _, ib, self.users_bias = self._bias_stats()
        if self.items_bias is None:
            self.items_bias = ib
        self.relationship_matrix_csr = self.relationship_matrix.tocsr()

    # ---- initialisation (mf.py:124-141) --------------------------------------------------------
    def init_feature_normal(self, mean=0.0, std=0.1):
        self.svd_u = np.random.normal(mean, std, [self.dimensionality, self.nbr_items])
        self.svd_v = np.random.normal(mean, std, [self.dimensionality, self.nbr_users])

    def init_user_features(self, user_index, mean=0.0, std=0.1):
        self.svd_v[:, user_index] = np.random.normal(mean, std, self.dimensionality)

    def init_item_features(self, item_index, mean=0.0, std=0.1):
        self.svd_u[:, item_index] = np.random.normal(mean, std, self.dimensionality)

    # ---- top-N (mf.py:144-193) ---------------------------------------------------------------------
    def _rated_items(self, user_index):
        """Row ids the reference reads from ``relationship_matrix_csc[:, user_index]`` (the matrix
        the subclass stored there; KMF keeps the transpose, so these are the user's items)."""
        col = self.relationship_matrix_csc[:, user_index].tocoo()
        return np.sort(col.row[col.data != 0]).astype(np.int32)

    # ---- resident model: the factors stay in HBM between calls ------------------------------------
    def invalidate_model(self):
        """Forget the device copy of the factors (call after editing svd_u / svd_v / the bias arrays
        element-wise; retraining and re-assignment are noticed without it)."""
        self._model_cache = None

    def _resident_model(self):
        """``mfrec_model`` of the current factors in identity layout, uploaded once and reused by
        predict / RMSE / top-N calls until the arrays change (their address, shape or sampled
        contents): ``test_predict_rating(nbr_samples=10)`` or one ``find_recommended_items`` call no
        longer moves 0.5 GB of factors at Netflix shape.  With more than one entry in
        ``options["devices"]`` it is a ``_native.ModelSet`` (one copy per listed device): batched top-N
        and predictions are split over them, with the one-device results."""
        devices = _serve_devices()
        key = (devices,) + tuple(_native.array_fingerprint(a)
                                 for a in (self.svd_u, self.svd_v, self.items_bias, self.users_bias))
        cached = getattr(self, '_model_cache', None)
        if cached is not None and cached[0] == key:
            return cached[1]
        k, ni = self.svd_u.shape
        args = (k, ni, self.svd_v.shape[1], self.svd_u, self.svd_v, self.items_bias, self.users_bias)
        model = _native.ModelSet(devices, *args) if devices else _native.Model(*args)
        self._model_cache = (key, model)
        return model

    def _rated_csr(self, users):
        """(indptr, items) of the rows ``relationship_matrix_csc[:, user]`` for a list of users."""
        m = self.relationship_matrix_csc
        indptr = np.zeros(len(users) + 1, dtype=np.int64)
        chunks = []
        for j, user in enumerate(users):
            a, b = m.indptr[user], m.indptr[user + 1]
            rows = m.indices[a:b][m.data[a:b] != 0]
            chunks.append(np.sort(rows))
            indptr[j + 1] = indptr[j] + rows.shape[0]
        flat = np.concatenate(chunks).astype(np.int32) if chunks else np.zeros(0, dtype=np.int32)
        return indptr, flat

    def _topn(self, user_index, n_candidates, nbr_recommendations, predictor):
        rated = self._rated_items(user_index)
        indptr = np.array([0, rated.shape[0]], dtype=np.int64)
        items, scores, counts = self._resident_model().topn(
            self.NATIVE_PREDICTORS[predictor], np.array([user_index], dtype=np.int32), n_candidates, indptr,
            rated, nbr_recommendations, self.overall_bias or 0.0, self.min_rating, self.max_rating)
        c = int(counts[0])
        return [int(i) for i in items[0, :c]], [float(s) for s in scores[0, :c]]

    def find_recommended_items_batch(self, user_indices, nbr_recommendations=5, predictor='predict'):
        """``find_recommended_items`` for MANY users in one device call (the all-users sweep on the
        tensor cores, ``mfrec_model_topn_sweep``): what ``metrics.precision_recall`` needs -- the
        reference calls ``find_recommended_items`` once per test user (metrics.py:104-107).  Same
        per-user results and the same RNG consumption as that loop.  Returns (items int32 [n, N]
        padded with -1, scores float64 [n, N], counts int32 [n])."""
        user_indices = np.asarray(user_indices, dtype=np.int32).reshape(-1)
        self.neighborhood = min([self.neighborhood, self.nbr_items])
        for _ in range(user_indices.shape[0]):
            self.get_items_subset(count=self.neighborhood)   # the reference draws (and ignores) a sample per call
        name = predictor if predictor in self.NATIVE_PREDICTORS else self._predict_alias(predictor)
        indptr, rated = self._rated_csr(user_indices)
        items, scores, counts, stats = self._resident_model().topn(
            self.NATIVE_PREDICTORS[name], user_indices, self.neighborhood, indptr, rated, nbr_recommendations,
            self.overall_bias or 0.0, self.min_rating, self.max_rating, sweep=True)
        self.last_topn_stats = stats
        return items, scores, counts

    def find_recommended_items(self, user_index=None, user_label=None, nbr_recommendations=5,
                               output_label=False, predictor='predict'):
        """Scores items for one user, drops the rated ones, returns the best N.  Reference quirks
        kept (SURVEY.md 3.4): the sampled item ids are drawn (the RNG advances) but the loop scores
        the enumeration index, i.e. items ``0 .. neighborhood-1``; the user's own index is added to
        the excluded item ids; exact zeros and NaNs are dropped."""
        if user_index is None:
            user_index = self.users_index[user_label]
        self.neighborhood = min([self.neighborhood, self.nbr_items])
        self.get_items_subset(count=self.neighborhood)
        name = predictor if predictor in self.NATIVE_PREDICTORS else self._predict_alias(predictor)
        items, scores = self._topn(user_index, self.neighborhood, nbr_recommendations, name)
        if output_label:
            items = [self.items_label[i] for i in items]
        return items, scores

    # ---- similarity in factor space (base.py:1294-1348 users, 1420-1466 items) ----------------------
    def _similarity_model(self, rows, method, tag):
        """Resident model whose "item" and "user" factors are both the prepared rows, so that one
        row of the similarity matrix is one top-N query.  cosine / Pearson: rows (centred for Pearson)
        scaled to unit length, score = dot.  euclidean: item side -2 x_i with bias |x_i|^2, user side
        x_q with bias |x_q|^2, so the linear predictor gives |x_i - x_q|^2.  Cached per (rows,
        method, devices): repeated queries upload nothing.  Several devices in ``options["devices"]``:
        a ``_native.ModelSet``, as for ``_resident_model``."""
        devices = _serve_devices()
        key = (tag, method, devices, _native.array_fingerprint(rows))
        cache = getattr(self, '_sim_cache', None)
        if cache is not None and cache[0] == key:
            return cache[1]
        x = np.array(rows, dtype=np.float64)
        if method == 'euclidean':
            sq = (x * x).sum(axis=1)
            args = (x.shape[1], x.shape[0], x.shape[0], np.ascontiguousarray(-2.0 * x.T), np.ascontiguousarray(x.T),
                    sq, sq)
        else:
            if method == 'pearson':
                x = x - x.mean(axis=1, keepdims=True)
            norm = np.sqrt((x * x).sum(axis=1, keepdims=True))
            x = np.divide(x, norm, out=np.zeros_like(x), where=norm > 0)
            xt = np.ascontiguousarray(x.T)                  # [d, n]: "item factors" and "user factors"
            args = (x.shape[1], x.shape[0], x.shape[0], xt, xt, None, None)
        model = _native.ModelSet(devices, *args) if devices else _native.Model(*args)
        self._sim_cache = (key, model)
        return model

    def _similar_rows_batch(self, rows, queries, nbr_recommendations, method, tag, skip_first=False):
        """Neighbours of every row in ``queries``: (ids [n, N], similarities [n, N], counts [n]), most
        similar first (euclidean: the reference sorts DISTANCES in descending order, i.e. farthest
        first -- kept).  The query row itself is excluded on the device.  skip_first: drop the head
        of each list (what the reference's ``similar_items`` does to a euclidean ranking, where the
        head is not the item itself)."""
        if method not in ('cosine', 'pearson', 'euclidean'):
            raise NotImplementedError("similarity method %r: 'cosine', 'pearson' and 'euclidean' run on the device" % method)
        n = rows.shape[0]
        N = n - 1 if nbr_recommendations == 'All' else int(nbr_recommendations)
        ask = max(min(N + (1 if skip_first else 0), n), 1)
        model = self._similarity_model(rows, method, tag)
        q = np.asarray(queries, dtype=np.int32).reshape(-1)
        predictor = 'predict_linear' if method == 'euclidean' else 'predict_dot'
        items, scores, counts = model.topn(predictor, q, n, None, None, ask, sweep=q.shape[0] >= 128)[:3]
        if method == 'euclidean':
            scores = np.sqrt(np.maximum(scores, 0.0))
        if skip_first:
            items, scores, counts = items[:, 1:], scores[:, 1:], np.maximum(counts - 1, 0)
        return items[:, :N], scores[:, :N], np.minimum(counts, N)

    def _similar_rows(self, rows, query, nbr_recommendations, similarity_threshold, similarities_output,
                      method, transform=None, tag='rows', skip_first=False):
        """Top neighbours of row ``query`` of ``rows`` ([n, d]), scored and ranked on the device by the
        top-N kernel (one row of a Gram matrix)."""
        items, scores, counts = self._similar_rows_batch(rows, [query], nbr_recommendations, method, tag, skip_first)
        c = int(counts[0])
        ids = [int(i) for i in items[0, :c]]
        sims = [float(v) for v in scores[0, :c]]
        if transform is not None:
            sims = [transform(v) for v in sims]
        if similarity_threshold:
            keep = [j for j, v in enumerate(sims) if v > similarity_threshold]
            ids, sims = [ids[j] for j in keep], [sims[j] for j in keep]
        return (ids, sims) if similarities_output else ids

    def similar_items(self, item_index, nbr_recommendations=2, similarity_threshold=False,
                      similarities_output=False, method='cosine'):
        return self._similar_rows(self.svd_u.T, item_index, nbr_recommendations, similarity_threshold,
                                  similarities_output, method, tag='items', skip_first=(method == 'euclidean'))

    def similar_items_batch(self, item_indices, nbr_recommendations=2, method='cosine'):
        """``similar_items`` for many items in one device call: (ids, similarities, counts)."""
        return self._similar_rows_batch(self.svd_u.T, item_indices, nbr_recommendations, method, 'items',
                                        skip_first=(method == 'euclidean'))

    def similar_users(self, user_index, nbr_recommendations=2, similarity_threshold=False,
                      similarities_output=False, method='pearson'):
        """User-user neighbours in factor space (base.py:1294-1348; the user itself is removed
        explicitly there, so no entry is skipped)."""
        return self._similar_rows(self.svd_v.T[:, 0:self.dimensionality], user_index, nbr_recommendations,
                                  similarity_threshold, similarities_output, method, tag='users')

    def similar_items_by_label(self, item_label, nbr_recommendations=2, similarity_threshold=False,
                               similarities_output=False, method='cosine'):
        out = self.similar_items(self.items_index[item_label], nbr_recommendations, similarity_threshold,
                                 True, method)
        labels = [self.items_label[i] for i in out[0]]
        return (labels, out[1]) if similarities_output else labels

    def _predict_alias(self, predictor):
        """'predict' is a class attribute aliasing one of the named predictors."""
        target = getattr(type(self), predictor)
        for name in self.NATIVE_PREDICTORS:
            if getattr(type(self), name, None) is target:
                return name
        raise KeyError(predictor)


def _serve_devices():
    """The devices predictions and top-N are served from: ``options["devices"]`` when it lists more than
    one (a ``_native.ModelSet``), else () (one ``_native.Model`` on the default context)."""
    devices = tuple(int(d) for d in options["devices"])
    return devices if len(devices) > 1 else ()


# ---- batched fold-in: argument checks shared by KMFRecommender and GDRecommender ------------------
def _fold_rows(indices, n):
    """The listed rows as int64: in [0, n) (IndexError) and distinct (ValueError)."""
    rows = np.asarray(indices).reshape(-1)
    if rows.shape[0] and not np.issubdtype(rows.dtype, np.integer):
        raise IndexError('row indices must be integers, got %s' % rows.dtype)
    rows = rows.astype(np.int64)
    bad = (rows < 0) | (rows >= n)
    if bad.any():
        raise IndexError('row %d is outside [0, %d)' % (rows[bad][0], n))
    if np.unique(rows).shape[0] != rows.shape[0]:
        raise ValueError('a row is listed more than once')
    return rows


def _fold_ratings(rows, col, n_other, ratings_index, ratings):
    """The ratings naming a listed row (column ``col``), in input order, checked like the single-row
    calls check theirs: int32 / float64 buffers (ValueError), the other index in [0, n_other)
    (IndexError)."""
    ids = np.nonzero(np.isin(ratings_index[:, col], rows))[0]
    idx = np.ascontiguousarray(ratings_index[ids, :])
    r = np.ascontiguousarray(ratings[ids])
    buffer_arg(idx, "ratings_index", np.int32, 2, writable=False)
    buffer_arg(r, "ratings", np.float64, 1, writable=False)
    other = idx[:, 1 - col]
    bad = (other < 0) | (other >= n_other)
    if bad.any():
        raise IndexError('rating (user, item) = (%d, %d) names no %s' % (idx[bad][0, 0], idx[bad][0, 1],
                                                                         'item' if col == 0 else 'user'))
    return idx, r
