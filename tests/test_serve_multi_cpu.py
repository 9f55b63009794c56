"""Serving from several shards (mfrec_model_topn_sweep_multi, mfrec_model_predict_multi,
_native.ModelSet) without a GPU: the symbols are declared and exported, and the recommenders route
batched calls to the shard set, single users to its first shard, and rebuild their cached models
when options["devices"] changes.  The native library and the device models are replaced by
recorders."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW = ("mfrec_model_topn_sweep_multi", "mfrec_model_predict_multi")


def test_new_entry_points_are_declared_and_exported():
    from mfrec_b200 import _native
    header = open(os.path.join(ROOT, "include", "mfrec_b200.h")).read()
    assert int(re.search(r"#define MFREC_B200_ABI_VERSION (\d+)", header).group(1)) >= 7
    for name in NEW:
        assert name in _native.EXPORTS
        assert re.search(r"\bint %s\(mfrec_ctx \*const \*ctxs, const mfrec_model \*const \*models, int n_shards," % name,
                         header), name
        assert hasattr(_native.lib(), name)
    assert hasattr(_native, "ModelSet") and hasattr(_native, "shard_contexts")


class _Ctx(object):
    count = 0

    def __init__(self, device):
        _Ctx.count += 1
        self.device, self.handle = device, 1000 + _Ctx.count


class _Model(object):
    """Stands in for _native.Model: records its construction and every call."""
    built = []

    def __init__(self, k, ni, nu, u=None, v=None, items_bias=None, users_bias=None, layout=None, ctx=None):
        self.k, self.ni, self.nu, self.ctx = k, ni, nu, ctx
        self.handle = 5000 + len(_Model.built)
        self.calls = []
        _Model.built.append(self)

    def topn(self, predictor, users, n_candidates, rated_indptr, rated_items, N, mu=0.0, min_rating=1.0,
             max_rating=5.0, sweep=False, out=None):
        self.calls.append(("topn", sweep))
        n = len(users)
        res = (np.full((n, N), -1, np.int32), np.zeros((n, N)), np.zeros(n, np.int32))
        return res + (np.zeros(8),) if sweep else res

    def predict(self, predictor, pairs, *a, **kw):
        self.calls.append(("predict",))
        return np.zeros(len(pairs)), None


class _Lib(object):
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append((name, args[2].value))   # (entry point, n_shards)
            return 0
        return call


@pytest.fixture()
def fakes(monkeypatch):
    from mfrec_b200 import _native
    from mfrec_b200.lib._buffers import options
    monkeypatch.setitem(options, "devices", [])
    _Model.built = []
    lib = _Lib()
    contexts = []

    def shard_contexts(devices):
        contexts.append(tuple(devices))
        return tuple(_Ctx(d) for d in devices)

    monkeypatch.setattr(_native, "Model", _Model)
    monkeypatch.setattr(_native, "lib", lambda: lib)
    monkeypatch.setattr(_native, "shard_contexts", shard_contexts)
    return options, lib, contexts


def _recommender():
    from mfrec_b200.recommendation import KMFRecommender
    rng = np.random.default_rng(1)
    nu, ni, k = 300, 200, 8
    rec = KMFRecommender(nu, ni, {'nbr_features': k})
    for _ in range(2000):
        rec.set_item_by_id(int(rng.integers(nu)), int(rng.integers(ni)), float(rng.integers(1, 6)))
    rec.svd_u, rec.svd_v = rng.normal(0, 0.1, (k, ni)), rng.normal(0, 0.1, (k, nu))
    rec.items_bias, rec.users_bias = np.zeros(ni), np.zeros(nu)
    rec.overall_bias = 3.0
    rec.relationship_matrix_csc = rec.relationship_matrix.T.tocsc()
    return rec


def test_one_device_keeps_the_single_model(fakes):
    from mfrec_b200 import _native
    options, lib, contexts = fakes
    rec = _recommender()
    for devices in ([], [3]):
        options["devices"] = devices
        m = rec._resident_model()
        assert type(m) is _Model and m.ctx is None            # default context, as before
    rec.find_recommended_items_batch(np.arange(150), 5, 'predict_linear')
    assert m.calls == [("topn", True)] and lib.calls == [] and contexts == []
    assert not isinstance(m, _native.ModelSet)


def test_batched_calls_go_to_the_set_single_users_to_shard_0(fakes):
    from mfrec_b200 import _native
    from mfrec_b200.recommendation import metrics
    options, lib, contexts = fakes
    rec = _recommender()
    options["devices"] = [2, 2, 2]
    ms = rec._resident_model()
    assert isinstance(ms, _native.ModelSet) and contexts == [(2, 2, 2)]
    assert len(ms.models) == 3 and len({id(m.ctx) for m in ms.models}) == 3   # a context per shard
    assert [m.ctx.device for m in ms.models] == [2, 2, 2]

    rec.find_recommended_items_batch(np.arange(150), 5, 'predict_linear')
    assert lib.calls == [("mfrec_model_topn_sweep_multi", 3)]
    assert rec.last_topn_stats.shape == (8,)
    rec.find_recommended_items(user_index=7, nbr_recommendations=5, predictor='predict_linear')
    assert ms.models[0].calls == [("topn", False)] and not ms.models[1].calls and not ms.models[2].calls

    held = np.c_[np.arange(40) % 300, np.arange(40) % 200, np.ones(40)]
    metrics.test_predict_rating(rec, held, nbr_samples=40, predictor='predict_linear')
    assert lib.calls[-1] == ("mfrec_model_predict_multi", 3)
    metrics.precision_recall(rec, held, nbr_recommendations=5, predictor='predict_linear')
    assert lib.calls[-1] == ("mfrec_model_topn_sweep_multi", 3)

    n_lib = len(lib.calls)
    rec.similar_items_batch(np.arange(200), nbr_recommendations=4)          # >= 128 queries: the sweep
    assert lib.calls[n_lib:] == [("mfrec_model_topn_sweep_multi", 3)]
    sim = rec._sim_cache[1]
    assert isinstance(sim, _native.ModelSet) and contexts[-1] == (2, 2, 2)
    rec.similar_items(5, nbr_recommendations=4)                             # one query: the first shard
    assert sim.models[0].calls == [("topn", False)] and not sim.models[1].calls
    assert rec._sim_cache[1] is sim                                         # cached
    assert rec._resident_model() is ms                                      # cached


def test_a_change_of_devices_rebuilds_the_cache(fakes):
    from mfrec_b200 import _native
    options, lib, contexts = fakes
    rec = _recommender()
    options["devices"] = [0, 1]
    a = rec._resident_model()
    assert rec._resident_model() is a
    options["devices"] = [1, 0]
    b = rec._resident_model()
    assert b is not a and isinstance(b, _native.ModelSet) and contexts[-1] == (1, 0)
    options["devices"] = []
    c = rec._resident_model()
    assert type(c) is _Model
    options["devices"] = [1, 0]
    assert rec._resident_model() is not b                                   # only the last key is kept
    rec.similar_items_batch(np.arange(200), nbr_recommendations=4)
    s1 = rec._sim_cache[1]
    options["devices"] = []
    rec.similar_items_batch(np.arange(200), nbr_recommendations=4)
    assert rec._sim_cache[1] is not s1 and type(rec._sim_cache[1]) is _Model


def test_a_failing_shard_fails_the_set(fakes, monkeypatch):
    from mfrec_b200 import _native

    class Failing(_Model):
        def __init__(self, *a, **kw):
            _Model.__init__(self, *a, **kw)
            if kw["ctx"].device == 9:
                raise MemoryError("shard out of memory")

    monkeypatch.setattr(_native, "Model", Failing)
    with pytest.raises(MemoryError):
        _native.ModelSet([1, 9, 1], 4, 10, 12, np.zeros((4, 10)), np.zeros((4, 12)))
