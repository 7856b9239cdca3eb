"""predictive_evaluation on the device (predict_batch): for CDAE and DMF the batched path returns the same dict as the
per-row loop over model.predict and as the oracle, from the same y_pred bit for bit; and predict() of a known user
with an unknown item is None (CDAE returned the user's whole score row)."""
import numpy as np
import pytest

import drecpy_b200 as drb
from oracle.predictive import predictive_evaluation_oracle

pytestmark = pytest.mark.gpu


def _split():
    u, i, v = drb.synthetic_interactions(120, 150, 4000, seed=3)
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=0.25, seed=4)
    train.assign_internal_ids()
    rng = np.random.default_rng(5)
    # unknown users (1000, 1001), items the model never saw (>= 1000), duplicate test rows
    su = np.concatenate([test.user, [1000, 1000, 1001], test.user[:15], rng.integers(1, 121, 25)])
    si = np.concatenate([test.item, [3, 4, 5], test.item[:15], rng.integers(1000, 1010, 25)])
    sv = np.concatenate([test.interaction, [5, 5, 1], rng.integers(1, 6, 40)]).astype(np.float64)
    order = rng.permutation(len(su))
    return train, drb.InteractionData(su[order], si[order], sv[order])


@pytest.fixture(scope='module')
def split():
    return _split()


@pytest.fixture(scope='module', params=['cdae', 'dmf'])
def model(request, split):
    train, _ = split
    if request.param == 'cdae':
        m = drb.CDAE(hidden_factors=50, seed=10, verbose=False)
    else:
        m = drb.DMF(user_factors=[16, 8], item_factors=[16, 8], seed=10, verbose=False)
    m.fit(train, epochs=3, batch_size=64)
    return m


GRID = [dict(), dict(count_none_predictions=True), dict(n_test_predictions=40),
        dict(count_none_predictions=True, n_test_predictions=333), dict(n_test_predictions=10 ** 6)]


@pytest.mark.parametrize('kw', GRID)
def test_fast_path_equals_general_path_and_oracle(model, split, kw):
    _, test = split
    metrics = [drb.RMSE(), drb.MSE(), drb.MAE()]
    tf, ts = {}, {}
    fast = drb.predictive_evaluation(model, test, metrics=metrics, timings=tf, **kw)
    slow = drb.predictive_evaluation(model, test, metrics=metrics, timings=ts, force_python=True, **kw)
    assert 'pair_kernel_ms' in tf and tf['pair_kernel_ms'] > 0            # the device path ran
    assert fast == slow
    assert np.array_equal(tf['y_pred'].view(np.uint64), ts['y_pred'].view(np.uint64))
    assert np.array_equal(tf['y_true'], ts['y_true'])
    want, yt, yp = predictive_evaluation_oracle(lambda u, i: model.predict(u, i, skip_errors=True), test.user.tolist(),
                                                test.item.tolist(), test.interaction.tolist(),
                                                metrics=('RMSE', 'MSE', 'MAE'), **kw)
    assert fast == want
    assert np.array_equal(tf['y_pred'].view(np.uint64), yp.view(np.uint64))


def test_train_evaluation(model, split):
    train, _ = split
    t = {}
    fast = drb.predictive_evaluation(model, timings=t)
    assert fast == drb.predictive_evaluation(model, train, force_python=True)
    assert t['n_rows'] == len(train)


def test_skip_errors_false(model, split):
    _, test = split
    with pytest.raises(AssertionError, match='was not found'):
        drb.predictive_evaluation(model, test, skip_errors=False)
    with pytest.raises(AssertionError, match='was not found'):
        drb.predictive_evaluation(model, test, skip_errors=False, force_python=True)


def test_unknown_item_predicts_none(model, split):
    train, _ = split
    user = train.raw_users[0]
    assert model.predict(user, 10 ** 6, skip_errors=True) is None
    assert model.predict(10 ** 6, train.raw_items[0], skip_errors=True) is None
    with pytest.raises(AssertionError, match=f'Item {10 ** 6} was not found.'):
        model.predict(user, 10 ** 6)
    p = model.predict(user, train.raw_items[0])
    assert np.ndim(p) == 0 and np.isfinite(p)
