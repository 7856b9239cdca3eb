"""recommendation_evaluation's per-user protocol (no GPU): the general path against the oracle restatement, with a
fake model whose recommend() is a deterministic function of (user, item)."""
import numpy as np
import pytest

import drecpy_b200 as drb
from oracle.recommendation import recommendation_evaluation_oracle


class FakeModel:
    """recommend() over the whole catalog with a fixed score per (user, item); unknown users assert, as
    DeepRecommenderABC.recommend does."""

    def __init__(self, train, threshold=0.001):
        self.interaction_dataset = self._data = train
        self.interaction_threshold = threshold
        self.n_items = train.count_unique('iid')

    def recommend(self, user_id, n=None, novelty=True, interaction_threshold=None, **kw):
        t = self._data
        uid = t.user_to_uid(user_id)
        assert uid is not None, f'User {user_id} was not found.'
        cand = set(range(self.n_items))
        if novelty:
            cand -= set(t.user_items(uid).tolist())
        r = sorted([(float((uid * 7919 + i * 104729) % 97) / 97.0, i) for i in cand], reverse=True)[:n]
        if interaction_threshold is not None:
            r = [x for x in r if x[0] >= interaction_threshold]
        return [(s, t.iid_to_item(i)) for s, i in r]


def _data(seed=0, float_values=False):
    rng = np.random.default_rng(seed)
    U, I = 40, 60
    tu, ti = rng.integers(0, U, 900), rng.integers(0, I, 900)
    tv = rng.integers(1, 6, 900).astype(np.float64)
    train = drb.InteractionData(tu, ti, tv)
    train.assign_internal_ids()
    # test rows: some users and items the model never saw, duplicate (user, item) rows, rows below the threshold
    su = np.concatenate([rng.integers(0, U, 300), [U + 1, U + 1, U + 2]])
    si = np.concatenate([rng.integers(0, I + 8, 300), [1, 2, 3]])
    sv = rng.integers(0, 6, len(su)).astype(np.float64)
    if float_values:
        sv = sv * 0.75 + rng.uniform(0, 0.2, len(sv))
    su = np.concatenate([su, su[:20]])                   # duplicate test rows
    si = np.concatenate([si, si[:20]])
    sv = np.concatenate([sv, sv[20:40]])
    return train, drb.InteractionData(su, si, sv)


def _oracle(m, test, thr, **kw):
    def rec(user, n, novelty, threshold):
        return [it for _, it in m.recommend(user, n=n, novelty=novelty, interaction_threshold=threshold)]
    return recommendation_evaluation_oracle(rec, test.user.tolist(), test.item.tolist(), test.interaction.tolist(),
                                            thr, **kw)


@pytest.mark.parametrize('k', [10, [1, 5, 20]])
@pytest.mark.parametrize('n_pos', [None, 1, 3])
@pytest.mark.parametrize('novelty', [False, True])
def test_general_path_matches_oracle(k, n_pos, novelty):
    train, test = _data()
    m = FakeModel(train, threshold=2.0)
    got = drb.recommendation_evaluation(m, test, k=k, n_pos_interactions=n_pos, novelty=novelty, seed=3)
    want = _oracle(m, test, 2.0, k=k, n_pos_interactions=n_pos, novelty=novelty, seed=3)
    assert got == want
    assert any(v != 0 for v in got.values())


@pytest.mark.parametrize('low', [0.3, 0.99, 2.0])
def test_low_prediction_threshold(low):
    train, test = _data(1)
    m = FakeModel(train, threshold=3.0)
    kw = dict(k=[3, 10], ignore_low_predictions_threshold=low, novelty=True)
    assert drb.recommendation_evaluation(m, test, **kw) == _oracle(m, test, 3.0, **kw)


def test_float_relevancies_and_n_test_users():
    train, test = _data(2, float_values=True)
    m = FakeModel(train, threshold=1.5)
    for n_users in (1, 7, None):
        kw = dict(k=[2, 8], n_test_users=n_users, n_pos_interactions=None)
        assert drb.recommendation_evaluation(m, test, **kw) == _oracle(m, test, 1.5, **kw)


def test_interaction_threshold_keyword_overrides_the_model():
    train, test = _data(3)
    m = FakeModel(train, threshold=0.001)
    got = drb.recommendation_evaluation(m, test, k=5, interaction_threshold=4.0)
    assert got == _oracle(m, test, 4.0, k=5)
    assert got != drb.recommendation_evaluation(m, test, k=5)


def test_users_without_positives_and_unknown_users_are_skipped():
    train, _ = _data(4)
    # user 0: rows all below the threshold (no positives: HitRatio / Recall skip it, Precision / NDCG count it);
    # user 999: unknown to the model; user 1: one positive on an item the model does not know
    test = drb.InteractionData(np.array([0, 0, 999, 1, 1]), np.array([3, 4, 3, 500, 5]),
                               np.array([1.0, 0.5, 5.0, 5.0, 1.0]))
    m = FakeModel(train, threshold=2.0)
    rec = []
    got = drb.recommendation_evaluation(m, test, k=[5, 50], record=rec)
    assert got == _oracle(m, test, 2.0, k=[5, 50])
    assert [r[0] for r in rec] == [0, 1]


def test_record_lists_each_users_recommendations():
    train, test = _data(5)
    m = FakeModel(train, threshold=2.0)
    rec, ref = [], []
    got = drb.recommendation_evaluation(m, test, k=[4, 7], n_pos_interactions=1, record=rec)
    assert got == _oracle(m, test, 2.0, k=[4, 7], n_pos_interactions=1, record=ref)
    assert len(rec) == len(ref) > 0
    for (u, c, r), (u2, c2, r2) in zip(rec, ref):
        assert u == u2 and sorted(c) == sorted(c2) and r == r2
        assert r == [it for _, it in m.recommend(u, n=7, novelty=False)]


def test_non_integer_raw_ids_take_the_python_candidate_path():
    train, test = _data(6)
    tr = drb.InteractionData(np.array([f'u{x}' for x in train.user]), np.array([f'i{x}' for x in train.item]),
                             train.interaction)
    tr.assign_internal_ids()
    te = drb.InteractionData(np.array([f'u{x}' for x in test.user]), np.array([f'i{x}' for x in test.item]),
                             test.interaction)
    m = FakeModel(tr, threshold=2.0)
    kw = dict(k=[3, 10], n_pos_interactions=2, seed=5)
    assert drb.recommendation_evaluation(m, te, **kw) == _oracle(m, te, 2.0, **kw)


def test_default_metrics_and_train_evaluation():
    train, _ = _data(7)
    m = FakeModel(train, threshold=2.0)
    got = drb.recommendation_evaluation(m, k=10)
    assert list(got) == ['Precision@10', 'Recall@10', 'HitRatio@10', 'NDCG@10']
    assert got == _oracle(m, train, 2.0, k=10)
    assert got == drb.recommendation_evaluation(m, train, k=10,
                                                metrics=[drb.Precision(), drb.Recall(), drb.HitRatio(), drb.NDCG()])
    assert drb.recommendation_evaluation(m, k=10, novelty=True) == _oracle(m, train, 2.0, k=10, novelty=True)


def test_argument_errors():
    train, test = _data(8)
    m = FakeModel(train)
    with pytest.raises(AssertionError, match=r'The number of test users \(0\) should be > 0.'):
        drb.recommendation_evaluation(m, test, n_test_users=0)
    with pytest.raises(AssertionError, match=r'The number of positive interactions \(0\) should be None or an integer '
                                             r'> 0.'):
        drb.recommendation_evaluation(m, test, n_pos_interactions=0)
    with pytest.raises(AssertionError, match=r'k \(0\) should be > 0.'):
        drb.recommendation_evaluation(m, test, k=[5, 0])
    with pytest.raises(AssertionError, match=r'Expected "metrics" argument to be a list'):
        drb.recommendation_evaluation(m, test, metrics=drb.NDCG())
    with pytest.raises(AssertionError, match=r'to be an instance of type RankingMetricABC'):
        drb.recommendation_evaluation(m, test, metrics=[1])
