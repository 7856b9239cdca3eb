"""recommendation_evaluation on the device (drb_eval_topk_metrics, eval_topk.cu): the fast path returns the same dict
as the per-user loop over model.recommend and as the oracle, and its per-user DCG / ideal DCG / hit counts are bit for
bit those of the host drb_eval_metrics on recommend_batch's lists (route A), for CDAE and DMF."""
import numpy as np
import pytest

import drecpy_b200 as drb
from drecpy_b200 import evaluation as E
from oracle.recommendation import recommendation_evaluation_oracle
from tools.bench_recommendation_evaluation import bitwise_equal, route_a

pytestmark = pytest.mark.gpu


def _split():
    u, i, v = drb.synthetic_interactions(70, 90, 2200, seed=3)
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=4, seed=4)
    train.assign_internal_ids()
    rng = np.random.default_rng(5)
    # unknown users (1000, 1001), items the model never saw (> 90), duplicate test rows, rows of every value
    su = np.concatenate([test.user, [1000, 1000, 1001], test.user[:15]])
    si = np.concatenate([test.item, [3, 4, 5], test.item[:15]])
    sv = np.concatenate([test.interaction, [5, 5, 1], rng.integers(1, 6, 15)]).astype(np.float64)
    extra = rng.integers(1, 71, 25)
    su, si = np.concatenate([su, extra]), np.concatenate([si, rng.integers(91, 99, 25)])
    sv = np.concatenate([sv, rng.integers(1, 6, 25)]).astype(np.float64)
    return train, drb.InteractionData(su, si, sv)


@pytest.fixture(scope='module')
def split():
    return _split()


@pytest.fixture(scope='module', params=['cdae', 'dmf'])
def model(request, split):
    train, _ = split
    if request.param == 'cdae':
        m = drb.CDAE(hidden_factors=32, seed=10, verbose=False, interaction_threshold=2.5)
        m.fit(train, epochs=3, batch_size=64)
    else:
        m = drb.DMF(user_factors=[16, 8], item_factors=[16, 8], seed=10, verbose=False, interaction_threshold=2.5)
        m.fit(train, epochs=3, batch_size=64)
    return m


def _oracle(m, test, **kw):
    def rec(user, n, novelty, threshold):
        return [it for _, it in m.recommend(user, n=n, novelty=novelty, interaction_threshold=threshold)]
    return recommendation_evaluation_oracle(rec, test.user.tolist(), test.item.tolist(), test.interaction.tolist(),
                                            m.interaction_threshold, **kw)


def _low(m, test, q):
    """A threshold on recommend()'s scores (CDAE: sigmoid outputs, DMF: rescaled to the rating range) that keeps a
    fraction of a list: the q-quantile of the first test user's top 40."""
    return float(np.quantile([s for s, _ in m.recommend(test.user[0].item(), n=40, novelty=False)], q))


def _check(m, test, **kw):
    kw = dict(kw)
    if 'low_q' in kw:
        kw['ignore_low_predictions_threshold'] = _low(m, test, kw.pop('low_q'))
    timings = {}
    fast = drb.recommendation_evaluation(m, test, timings=timings, **kw)
    assert 'per_user' in timings                                   # the device path ran
    slow = drb.recommendation_evaluation(m, test, force_python=True, **kw)
    assert fast == slow
    okw = {x: kw[x] for x in ('k', 'n_pos_interactions', 'novelty', 'ignore_low_predictions_threshold', 'seed',
                              'n_test_users') if x in kw}
    if test is not None:
        assert fast == _oracle(m, test, **okw)
    return fast, timings['per_user']


GRID = [dict(k=10), dict(k=[1, 5, 20]), dict(k=[3, 10], n_pos_interactions=1, seed=7),
        dict(k=[2, 40], n_pos_interactions=3, novelty=True), dict(k=[5, 15], novelty=True, n_test_users=9),
        dict(k=[4, 12], low_q=0.3), dict(k=[4, 12], n_pos_interactions=1, novelty=True, low_q=0.8)]


@pytest.mark.parametrize('kw', GRID, ids=[str(g) for g in GRID])
def test_fast_path_equals_general_path_and_oracle(model, split, kw):
    res, _ = _check(model, split[1], **kw)
    assert any(v != 0 for v in res.values())


def test_float_relevancies(model, split):
    _, test = split
    rng = np.random.default_rng(9)
    t = drb.InteractionData(test.user, test.item, test.interaction * 0.7 + rng.uniform(0, 0.3, len(test)))
    _check(model, t, k=[3, 30], novelty=True)


def test_chunks_smaller_than_the_user_count(model, split):
    a, _ = _check(model, split[1], k=[5, 10], chunk=7)
    assert a == drb.recommendation_evaluation(model, split[1], k=[5, 10])


def test_lists_shorter_than_k(model, split):
    # novelty leaves about 60 unseen items of 90: the top-2000 lists are shorter than k
    _, pu = _check(model, split[1], k=[5, 2000], novelty=True)
    assert (pu['n_rec'][:, 1] < 2000).all() and (pu['n_rec'][:, 1] > 0).any()


def test_threshold_between_a_float32_score_and_the_next_double(model, split):
    _, test = split
    user = test.user[0].item()
    scores = [s for s, _ in model.recommend(user, n=20, novelty=False)]
    s = scores[7]
    for low in (float(s), float(np.nextafter(np.float64(s), np.inf)), float(np.nextafter(np.float64(s), -np.inf))):
        res, pu = _check(model, test, k=[5, 20], ignore_low_predictions_threshold=low)


def test_per_user_values_bitwise_equal_host_metrics(model, split):
    _, test = split
    for kw in (dict(k=[3, 10, 25]), dict(k=[5, 50], n_pos_interactions=1, novelty=True, seed=2),
               dict(k=[5, 20], ignore_low_predictions_threshold=_low(model, test, 0.5), novelty=True)):
        t = {}
        res = drb.recommendation_evaluation(model, test, timings=t, **kw)
        pu = t['per_user']
        ref, ref_pu = route_a(model, test, pu['users'], kw['k'], n_pos=kw.get('n_pos_interactions'),
                              novelty=kw.get('novelty', False), low=kw.get('ignore_low_predictions_threshold'),
                              seed=kw.get('seed', 0))
        assert res == ref
        assert bitwise_equal(pu, ref_pu)


def test_train_evaluation_bitwise(model):
    # ds_test=None: the evaluated set of a user is its whole training row, longer than max(k)
    t = {}
    res = drb.recommendation_evaluation(model, None, k=[5, 20], timings=t)
    pu = t['per_user']
    ref, ref_pu = route_a(model, None, pu['users'], [5, 20])
    assert res == ref and bitwise_equal(pu, ref_pu)
    assert res == drb.recommendation_evaluation(model, None, k=[5, 20], force_python=True)
    assert (pu['idcg'][:, 1] > 0).all()


def test_k_beyond_the_top_k_limit_takes_the_general_path(model, split, monkeypatch):
    _, test = split

    def no_fast(*a, **k):
        raise AssertionError('fast path taken')
    ref = drb.recommendation_evaluation(model, test, k=[5, 2049], n_test_users=6)
    monkeypatch.setattr(E, '_fast_recommendation_evaluation', no_fast)
    assert drb.recommendation_evaluation(model, test, k=[5, 2049], n_test_users=6) == ref
    assert ref == _oracle(model, test, k=[5, 2049], n_test_users=6)


@pytest.mark.parametrize('which', ['cdae', 'dmf'])
def test_epoch_callback(split, which):
    train, test = split
    stored = []

    def cb(m):
        stored.append(drb.recommendation_evaluation(m, test, k=10))
        return stored[-1]
    if which == 'cdae':
        m = drb.CDAE(hidden_factors=16, seed=3, verbose=True)
    else:
        m = drb.DMF(user_factors=[8], item_factors=[8], seed=3, verbose=True)
    m.fit(train, epochs=4, batch_size=64, epoch_callback_fn=cb, epoch_callback_freq=2)
    assert len(stored) == 3          # before training, epochs 2 and 4
    assert stored[-1] == drb.recommendation_evaluation(m, test, k=10)
    assert stored[-1] == drb.recommendation_evaluation(m, test, k=10, force_python=True)


def test_full_size_cdae_equals_route_a():
    u, i, v = drb.synthetic_interactions(138493, 26744, 20_000_000, seed=10, zipf_a=1.0)
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=1, seed=10, max_concurrent_threads=16)
    train.assign_internal_ids()
    m = drb.CDAE(hidden_factors=200, seed=10, verbose=False, rng_mode='philox')
    m.fit(train, epochs=1, batch_size=4096)
    t = {}
    res = drb.recommendation_evaluation(m, test, k=[10, 100], novelty=True, timings=t)
    pu = t['per_user']
    assert len(pu['users']) == len(np.unique(test.user))
    ref, ref_pu = route_a(m, test, pu['users'], [10, 100], novelty=True)
    assert res == ref and bitwise_equal(pu, ref_pu)
    assert res['HitRatio@100'] > 0
