"""recommend_batch (recommender.py) on a model without a GPU: a fake DeepRecommenderABC whose scores are a fixed
function of (user, item), ranked by the base class's own recommend() -> _rank -> _rank_batch route on one side and by
the fake's topk_batch on the other.  Covers the raw-id mapping both ways, the threshold cut, padding, chunking and the
unknown-user assertion."""
import numpy as np
import pytest

import drecpy_b200 as drb
from drecpy_b200.recommender import DeepRecommenderABC


class FakeTopkModel(DeepRecommenderABC):
    def __init__(self, data):
        super().__init__(verbose=False)
        self._data = data
        self.n_users = data.count_unique('uid')
        self.n_items = data.count_unique('iid')
        self.min_interaction, self.max_interaction = 0, 5
        self.fitted = True
        self.calls = []

    def _pre_fit(self, *a, **k): pass

    def _train_step(self, *a, **k): pass

    def _predict(self, uid, iid, **kwds):
        return self._scores(uid)[iid]

    def _scores(self, uid):
        # a few exact ties per user (values on a coarse grid), float32 as the library returns them
        return (np.float32(((uid * 7919 + np.arange(self.n_items) * 104729) % 31) / 31.0 * 5.0)).astype(np.float32)

    def _ranked(self, uid, cand, novelty):
        cand = set(int(c) for c in cand)
        if novelty:
            cand -= set(self._data.user_items(uid).tolist())
        p = self._scores(uid)
        return sorted(((p[i], i) for i in cand), reverse=True)

    def _rank_batch(self, uids, cand, cand_count, novelty):
        n, max_c = cand.shape
        oi = np.zeros((n, max_c), np.int32)
        os_ = np.zeros((n, max_c), np.float32)
        on = np.zeros(n, np.int32)
        for r, uid in enumerate(uids):
            ranked = self._ranked(int(uid), cand[r, :cand_count[r]], novelty)
            on[r] = len(ranked)
            for j, (s, i) in enumerate(ranked):
                os_[r, j], oi[r, j] = s, i
        return oi, os_, on

    def topk_batch(self, uids, k, novelty=True, return_device=False):
        self.calls.append(len(uids))
        n = len(uids)
        oi = np.zeros((n, k), np.int32)
        os_ = np.zeros((n, k), np.float32)
        on = np.zeros(n, np.int32)
        for r, uid in enumerate(np.asarray(uids).tolist()):
            p = self._scores(uid)
            alive = np.ones(self.n_items, bool)
            if novelty:
                alive[self._data.user_items(uid)] = False
            idx = np.flatnonzero(alive)
            order = np.lexsort((-idx, -p[idx]))[:k]      # score desc, then iid desc
            on[r] = len(order)
            oi[r, :len(order)], os_[r, :len(order)] = idx[order], p[idx][order]
        return oi, os_, on


def _data():
    u, i, v = drb.synthetic_interactions(60, 80, 1500, seed=3)
    # raw ids that are not the internal ones: users offset and reversed, items spread out
    ds = drb.InteractionData(1000 - u, 7 * i + 3, v)
    ds.assign_internal_ids()
    return ds


def _recommend_rows(m, users, n, novelty, thr):
    return [m.recommend(u, n=n, novelty=novelty, interaction_threshold=thr) for u in users]


@pytest.mark.parametrize('novelty', [True, False])
@pytest.mark.parametrize('thr', [None, 4.5])
def test_recommend_batch_rows_equal_recommend(novelty, thr):
    m = FakeTopkModel(_data())
    users = np.array(m._data.raw_users)[::-1][:40]
    items, scores, counts = m.recommend_batch(users, n=25, novelty=novelty, interaction_threshold=thr)
    assert items.shape == (40, 25) and scores.shape == (40, 25) and counts.shape == (40,)
    assert items.dtype == np.int64
    for r, want in enumerate(_recommend_rows(m, users, 25, novelty, thr)):
        assert counts[r] == len(want)
        assert items[r, :counts[r]].tolist() == [it for _, it in want]        # raw item ids
        assert scores[r, :counts[r]].tolist() == [float(s) for s, _ in want]
        assert (items[r, counts[r]:] == -1).all() and np.isnan(scores[r, counts[r]:]).all()
    if thr is not None:
        assert (counts < 25).any() and (scores[~np.isnan(scores)] >= thr).all()


def test_recommend_batch_padding_when_few_items_are_left():
    m = FakeTopkModel(_data())
    user = m._data.raw_users[0]
    left = m.n_items - len(m._data.user_items(m._data.user_to_uid(user)))
    items, scores, counts = m.recommend_batch([user], n=m.n_items, novelty=True)
    assert counts[0] == left < m.n_items
    assert (items[0, left:] == -1).all() and np.isnan(scores[0, left:]).all()
    items, _, counts = m.recommend_batch([user], n=m.n_items, novelty=False)
    assert counts[0] == m.n_items and (items[0] >= 0).all()


def test_recommend_batch_chunks():
    m = FakeTopkModel(_data())
    users = m._data.raw_users
    whole = m.recommend_batch(users, n=7)
    m.calls.clear()
    parts = m.recommend_batch(users, n=7, chunk=16)
    assert m.calls == [16] * (len(users) // 16) + ([len(users) % 16] if len(users) % 16 else [])
    for a, b in zip(whole, parts):
        np.testing.assert_array_equal(a, b)


def test_recommend_batch_errors():
    m = FakeTopkModel(_data())
    with pytest.raises(AssertionError, match='User 123456 was not found.'):
        m.recommend_batch([m._data.raw_users[0], 123456], n=5)
    for n in (0, 2049):
        with pytest.raises(ValueError, match=r'n must be in \[1, 2048\]'):
            m.recommend_batch([m._data.raw_users[0]], n=n)
    assert m.calls == []
