"""predictive_evaluation without a GPU: the per-row path and the batched path (driven by a duck-typed model with
predict_batch) against the oracle restatement, and the regression metrics against sklearn."""
import numpy as np
import pytest

import drecpy_b200 as drb
from oracle.predictive import predictive_evaluation_oracle


class StubModel:
    """predict() is a float32 function of the internal ids; unknown ids assert unless skip_errors (then None), as
    DeepRecommenderABC.predict does."""

    def __init__(self, train):
        self.interaction_dataset = self._data = train

    @staticmethod
    def _score(uid, iid):
        return (np.asarray((uid * 7919 + iid * 104729) % 97, np.float32) / np.float32(97)) * np.float32(5)

    def predict(self, user_id, item_id, skip_errors=False, **kw):
        t = self._data
        uid, iid = t.user_to_uid(user_id), t.item_to_iid(item_id)
        assert skip_errors or uid is not None, f'User {user_id} was not found.'
        assert skip_errors or iid is not None, f'Item {item_id} was not found.'
        if uid is None or iid is None:
            return None
        return self._score(np.int64(uid), np.int64(iid))[()]


class BatchStubModel(StubModel):
    """The same model with the batched interface of CDAE / DMF (predict_batch over raw ids, NaN for None)."""

    def __init__(self, train):
        super().__init__(train)
        self.batch_calls = []

    def _pair_ids(self, user_ids, item_ids):
        return (self._data.users_to_uids(user_ids).astype(np.int32), self._data.items_to_iids(item_ids).astype(np.int32))

    def predict_batch(self, user_ids, item_ids, skip_errors=False, chunk=1 << 22):
        self.batch_calls.append(len(user_ids))
        uids, iids = self._pair_ids(user_ids, item_ids)
        bad = (uids < 0) | (iids < 0)
        assert skip_errors or not bad.any()
        out = self._score(uids.astype(np.int64), iids.astype(np.int64))
        out[bad] = np.nan
        return out


def _data(seed=0, strings=False):
    rng = np.random.default_rng(seed)
    U, I = 30, 50
    tu, ti = rng.integers(0, U, 600), rng.integers(0, I, 600)
    tv = rng.integers(1, 6, 600).astype(np.float64)
    su = np.concatenate([rng.integers(0, U + 4, 400)])              # some users and items the model never saw
    si = np.concatenate([rng.integers(0, I + 6, 400)])
    sv = rng.uniform(0, 5, 400)
    if strings:
        tu, ti = np.array([f'u{x}' for x in tu]), np.array([f'i{x}' for x in ti])
        su, si = np.array([f'u{x}' for x in su]), np.array([f'i{x}' for x in si])
    train = drb.InteractionData(tu, ti, tv)
    train.assign_internal_ids()
    return train, drb.InteractionData(su, si, sv)


def _oracle(m, test, **kw):
    return predictive_evaluation_oracle(lambda u, i: m.predict(u, i, skip_errors=True), test.user.tolist(),
                                        test.item.tolist(), test.interaction.tolist(), **kw)


@pytest.mark.parametrize('count_none', [False, True])
@pytest.mark.parametrize('n_test', [None, 1, 17, 10_000])
@pytest.mark.parametrize('cls', [StubModel, BatchStubModel])
def test_matches_oracle(cls, count_none, n_test):
    train, test = _data()
    m = cls(train)
    metrics = [drb.RMSE(), drb.MSE(), drb.MAE()]
    timings = {}
    got = drb.predictive_evaluation(m, test, count_none_predictions=count_none, n_test_predictions=n_test,
                                    metrics=metrics, timings=timings)
    want, yt, yp = _oracle(m, test, count_none_predictions=count_none, n_test_predictions=n_test,
                           metrics=('RMSE', 'MSE', 'MAE'))
    assert got == want and list(got) == ['RMSE', 'MSE', 'MAE']
    assert timings['y_true'].dtype == timings['y_pred'].dtype == np.float64
    assert np.array_equal(timings['y_true'], yt)
    assert np.array_equal(timings['y_pred'].view(np.uint64), yp.view(np.uint64))
    if cls is BatchStubModel:
        assert len(m.batch_calls) == 1
        assert timings['n_rows'] == len(yt)


def test_batched_path_equals_per_row_path():
    train, test = _data(1)
    for kw in (dict(), dict(count_none_predictions=True), dict(n_test_predictions=33),
               dict(count_none_predictions=True, n_test_predictions=5)):
        a, b = {}, {}
        fast = drb.predictive_evaluation(BatchStubModel(train), test, timings=a, **kw)
        slow = drb.predictive_evaluation(BatchStubModel(train), test, timings=b, force_python=True, **kw)
        assert fast == slow
        assert np.array_equal(a['y_pred'].view(np.uint64), b['y_pred'].view(np.uint64))
        assert 'predict_batch_s' in a and 'predict_batch_s' not in b


def test_none_predictions_skipped_or_counted_as_zero():
    train, _ = _data(2)
    u0, i0 = train.raw_users[0], train.raw_items[0]
    test = drb.InteractionData(np.array([u0, 999, u0]), np.array([i0, i0, 999]), np.array([4.0, 3.0, 2.0]))
    p = float(StubModel(train).predict(u0, i0))
    got = drb.predictive_evaluation(StubModel(train), test, metrics=[drb.MSE()])
    assert got == {'MSE': round((4.0 - p) ** 2, 4)}
    got = drb.predictive_evaluation(StubModel(train), test, metrics=[drb.MSE()], count_none_predictions=True)
    assert got == {'MSE': round(((4.0 - p) ** 2 + 9.0 + 4.0) / 3, 4)}


def test_train_evaluation_when_ds_test_is_none():
    train, _ = _data(3)
    for cls in (StubModel, BatchStubModel):
        m = cls(train)
        assert drb.predictive_evaluation(m) == _oracle(m, train)[0]
        assert drb.predictive_evaluation(m) == drb.predictive_evaluation(m, train)


def test_string_raw_ids():
    train, test = _data(4, strings=True)
    for cls in (StubModel, BatchStubModel):
        m = cls(train)
        got = drb.predictive_evaluation(m, test, count_none_predictions=True, n_test_predictions=150)
        assert got == _oracle(m, test, count_none_predictions=True, n_test_predictions=150)[0]


def test_skip_errors_false_raises_predicts_assertion():
    train, _ = _data(5)
    u0, i0 = train.raw_users[0], train.raw_items[0]
    test = drb.InteractionData(np.array([u0, u0, 999]), np.array([i0, 777, i0]), np.array([1.0, 2.0, 3.0]))
    for cls in (StubModel, BatchStubModel):
        with pytest.raises(AssertionError, match='Item 777 was not found.'):
            drb.predictive_evaluation(cls(train), test, skip_errors=False)
        # the cap is reached before the unknown item: nothing raises
        assert drb.predictive_evaluation(cls(train), test, skip_errors=False, n_test_predictions=1) == \
            _oracle(cls(train), test, n_test_predictions=1)[0]
    test = drb.InteractionData(np.array([999, u0]), np.array([i0, i0]), np.array([1.0, 2.0]))
    for cls in (StubModel, BatchStubModel):
        with pytest.raises(AssertionError, match='User 999 was not found.'):
            drb.predictive_evaluation(cls(train), test, skip_errors=False)


def test_argument_errors():
    train, test = _data(6)
    m = StubModel(train)
    with pytest.raises(AssertionError, match=r'The number of test predictions \(0\) should be > 0.'):
        drb.predictive_evaluation(m, test, n_test_predictions=0)
    with pytest.raises(AssertionError, match=r'Expected "metrics" argument to be a list'):
        drb.predictive_evaluation(m, test, metrics=drb.RMSE())
    with pytest.raises(AssertionError, match=r'to be an instance of type PredictiveMetricABC'):
        drb.predictive_evaluation(m, test, metrics=[1])
    assert list(drb.predictive_evaluation(m, test)) == ['RMSE', 'MSE']


@pytest.mark.parametrize('seed', range(5))
def test_metrics_match_sklearn(seed):
    sk = pytest.importorskip('sklearn.metrics')
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 5000))
    y_true = rng.uniform(-3, 8, n)
    y_pred = rng.normal(2, 3, n).astype(np.float32 if seed % 2 else np.float64)
    assert drb.MSE()(y_true, y_pred) == pytest.approx(sk.mean_squared_error(y_true, y_pred), rel=1e-12)
    assert drb.MAE()(y_true, y_pred) == pytest.approx(sk.mean_absolute_error(y_true, y_pred), rel=1e-12)
    assert drb.RMSE()(y_true, y_pred) == pytest.approx(np.sqrt(sk.mean_squared_error(y_true, y_pred)), rel=1e-12)
    assert (drb.RMSE().name, drb.MSE().name, drb.MAE().name) == ('RMSE', 'MSE', 'MAE')
