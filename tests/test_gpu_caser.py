"""Caser on the GPU against the float64 oracle (oracle/caser.py): the device batch, one step's loss and raw gradients,
20 steps of two update rules, graph replay, bit-identical scores across every scoring entry point, the evaluation
protocols, save / load, reverts and the size checks."""
import os

import numpy as np
import pytest

import drecpy_b200 as drb
from oracle import caser as oc

pytestmark = pytest.mark.gpu

L, T, D, NV, NH, NEG, B = 5, 3, 50, 4, 16, 3, 48


def _data(seed=3, U=70, I=150, n=3000):
    u, i, v = drb.synthetic_interactions(U, I, n, seed=seed)
    ts = np.random.default_rng(seed).integers(0, 10 ** 6, len(u))
    return drb.InteractionData(u, i, v, timestamp=ts)


def _fit(ds, epochs=0, opt=None, L=L, T=T, d=D, n_v=NV, n_h=NH, rate=0.5, init=None, **kw):
    m = drb.Caser(L=L, T=T, d=d, n_v=n_v, n_h=n_h, dropout_rate=rate, seed=11, verbose=False, **kw)
    m.fit(ds, epochs=epochs, batch_size=B, neg_ratio=NEG, reg_rate=1e-3, optimizer=opt, init_weights=init)
    return m


def _oracle_of(m, opt=None):
    w = {k: ([x.detach().cpu().numpy() for x in v] if isinstance(v, list) else v.detach().cpu().numpy())
         for k, v in m.weights().items()}
    return oc.CaserOracle(w, opt)


def _seq(m):
    ds = m._data
    indptr, seq = oc.sequences(ds.uid, ds.iid, ds.interaction, m.n_users, m.interaction_threshold, ds.timestamp)
    return indptr, seq, oc.window_offsets(indptr, m.L, m.T)


def _oracle_batch(m, step):
    indptr, seq, win = _seq(m)
    return oc.sample_batch(indptr, seq, win, m._data.csr()[:2], m.n_items, m.L, m.T, m.neg_ratio, B, m.philox_seed(), step)


@pytest.fixture(scope='module')
def ds():
    return _data()


def test_device_batch_equals_oracle(ds):
    m = _fit(ds)
    for step in (1, 2, 9):
        m._step = step
        m._train_step(B, 1e-3)
        users, items = m.last_batch()
        ou, oi = _oracle_batch(m, step)
        assert np.array_equal(users[:B], ou)
        assert np.array_equal(items[:B], oi)


@pytest.mark.parametrize('shape', [dict(), dict(L=3, T=1, d=20, n_v=2, n_h=3, rate=0.0)], ids=['default', 'odd'])
def test_one_step_loss_and_gradients(ds, shape):
    m = _fit(ds, **shape)
    o = _oracle_of(m)
    m._step = 1
    loss = m._train_step(B, 1e-3, want_loss=True)
    users, items = _oracle_batch(m, 1)
    F = m.n_v * m.d + m.n_h * m.L
    scale = oc.dropout_scale(F, B, m.philox_seed(), 1, m.dropout_rate)
    want, g, _ = o.loss_and_grads(users, items, m.L, m.T, scale, 1e-3)
    assert abs(loss - want) <= 2e-5 * abs(want)
    got = m.weights(m._grads)
    for k, v in got.items():
        for j, x in enumerate(v if isinstance(v, list) else [v]):
            ref = g[k][j] if isinstance(v, list) else g[k]
            err = np.abs(x.cpu().numpy() - ref).max()
            scale_ = max(np.abs(ref).max(), 1e-12)
            assert err <= 2e-4 * scale_, (k, j, err, scale_)


@pytest.mark.parametrize('opt', [None, {'name': 'RMSprop', 'learning_rate': 1e-3}], ids=['adam', 'rmsprop'])
def test_twenty_steps_track_the_oracle(ds, opt):
    m = _fit(ds, opt=opt)
    o = _oracle_of(m, opt if opt else {'name': 'Adam', 'learning_rate': 1e-3})
    F = m.n_v * m.d + m.n_h * m.L
    for s in range(1, 21):
        m._step = s
        loss = m._train_step(B, 1e-3, want_loss=True)
        users, items = _oracle_batch(m, s)
        want = o.step(users, items, m.L, m.T, oc.dropout_scale(F, B, m.philox_seed(), s, m.dropout_rate), 1e-3)
        assert abs(loss - want) <= 1e-3 * abs(want), (s, loss, want)
    for k in ('E', 'W2', 'fc', 'Fv'):
        got, ref = m.weights()[k].cpu().numpy(), o.w[k]
        assert np.abs(got - ref).max() <= 1e-3 * np.abs(ref).max(), k


def test_graph_replay_equals_plain_launches(ds, monkeypatch):
    a = _fit(ds)
    monkeypatch.setenv('DRB_GRAPH', '0')
    b = _fit(ds)
    for s in range(1, 6):
        for m in (a, b):
            m._step = s
            m._train_step(B, 1e-3)
    la, lb = a.launch_count(), b.launch_count()
    assert la > 0 and lb > 0
    assert np.array_equal(a.last_batch()[1], b.last_batch()[1])
    pa, pb = a._params.cpu().numpy(), b._params.cpu().numpy()
    assert np.abs(pa - pb).max() <= 1e-5 * np.abs(pb).max()


@pytest.fixture(scope='module')
def fitted(ds):
    return _fit(ds, epochs=5)


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


def test_scoring_entry_points_agree_bitwise(fitted):
    m = fitted
    data = m._data
    users = data.raw_users[:12]
    items = data.raw_items
    rows = {u: m._predict(data.user_to_uid(u)) for u in users}
    indptr, seq, _ = _seq(m)
    ref = _oracle_of(m).predict_all(indptr, seq, [data.user_to_uid(u) for u in users])
    for r, u in enumerate(users):
        np.testing.assert_allclose(rows[u], ref[r], rtol=1e-5, atol=1e-6)
        assert _bits(m.predict(u, items[3])) == _bits(rows[u][3])
        pb = m.predict_batch(np.full(len(items), u), items)
        assert np.array_equal(_bits(pb), _bits(rows[u]))
        ranked = m.rank(u, items, novelty=False)
        for s, it in ranked:
            assert _bits(s) == _bits(rows[u][data.item_to_iid(it)])
        rec = m.recommend(u, n=30, novelty=True)
        assert [it for _, it in rec] == [it for _, it in ranked if it not in set(data.item[data.user == u].tolist())][:30]
        assert all(_bits(s) == _bits(rows[u][data.item_to_iid(it)]) for s, it in rec)
    ri, rs, rn = m.recommend_batch(users, n=30)
    ti, ts, tn = m.topk_batch(np.array([data.user_to_uid(u) for u in users], np.int32), 30)
    for r, u in enumerate(users):
        rec = m.recommend(u, n=30)
        assert ri[r, :rn[r]].tolist() == [it for _, it in rec]
        assert np.array_equal(_bits(rs[r, :rn[r]]), _bits([s for s, _ in rec]))
        assert np.array_equal(_bits(ts[r, :tn[r]]), _bits(rs[r, :rn[r]]))


def test_evaluation_protocols_equal_general_path(ds):
    tr, te = drb.leave_k_out(ds, k=3, seed=2)
    m = _fit(tr, epochs=4)
    kw = dict(k=[1, 5, 10], seed=3)
    assert drb.ranking_evaluation(m, te, n_neg_interactions=20, **kw) == \
        drb.ranking_evaluation(m, te, n_neg_interactions=20, force_python=True, **kw)
    assert drb.recommendation_evaluation(m, te, **kw) == drb.recommendation_evaluation(m, te, force_python=True, **kw)
    assert drb.predictive_evaluation(m, te) == drb.predictive_evaluation(m, te, force_python=True)


def test_save_load_and_revert_restore_scores(ds, tmp_path, fitted):
    m = fitted
    u = m._data.raw_users[4]
    row = m._predict(m._data.user_to_uid(u))
    path = os.path.join(tmp_path, 'caser.joblib')
    m.save(path)
    m2 = drb.Caser.load(path)
    assert np.array_equal(_bits(m2._predict(m2._data.user_to_uid(u))), _bits(row))

    class StopAt2:
        def compute(self, losses, results, epochs):
            return 2

        def stop_training(self, e, best, epochs):
            return e >= 4
    m3 = drb.Caser(seed=11, verbose=False)
    m3.fit(ds, epochs=4, batch_size=B, neg_ratio=NEG, early_stopping_rule=StopAt2(), early_stopping_freq=2)
    snap = m3.epoch_weights[2].to(m3._params.device)
    assert m3._params.equal(snap)
    uid = m3._data.user_to_uid(u)
    before = m3._predict(uid)
    m3._params.copy_(snap)
    assert np.array_equal(_bits(m3._predict(uid)), _bits(before))


def test_out_of_range_sizes_raise(ds):
    for kw in (dict(L=0), dict(L=17), dict(T=0), dict(T=33), dict(d=0), dict(d=300), dict(n_v=0), dict(n_h=65),
               dict(d=256, n_h=64), dict(dropout_rate=1.0)):
        with pytest.raises(ValueError):
            drb.Caser(**kw)
    with pytest.raises(ValueError, match='no_such_column'):
        drb.Caser(sort_column='no_such_column', verbose=False).fit(ds, epochs=1)
    with pytest.raises(ValueError, match='L \\+ T'):
        drb.Caser(L=16, T=32, d=8, n_v=1, n_h=2, verbose=False, sort_column=None).fit(_data(U=70, I=150, n=700), epochs=1)
