"""predict_batch (drb_cdae_predict_pairs / drb_dmf_predict_pairs, predict.cu) against the predict() loop: every element
bit for bit and with predict()'s dtype, for CDAE and DMF, across input shapes, training, weight reverts and save / load,
and at the full ml-20m shape."""
import numpy as np
import pytest

import drecpy_b200 as drb
from drecpy_b200 import _lib

pytestmark = pytest.mark.gpu

U, I = 1500, 400           # more users than max_batch (min(1024, n_users)): several user blocks per call

MODELS = {
    'cdae32': lambda: drb.CDAE(hidden_factors=32, seed=3, verbose=False),
    'cdae50': lambda: drb.CDAE(hidden_factors=50, seed=3, verbose=False),       # ld padded to 52
    'cdae200': lambda: drb.CDAE(hidden_factors=200, seed=3, verbose=False),
    'dmf16_8': lambda: drb.DMF(user_factors=[16, 8], item_factors=[16, 8], seed=3, verbose=False),
    'dmf64_32': lambda: drb.DMF(seed=3, verbose=False),
    'dmf3': lambda: drb.DMF(user_factors=[24, 16, 8], item_factors=[32, 12, 8], seed=3, verbose=False),
}


@pytest.fixture(scope='module')
def train():
    u, i, v = drb.synthetic_interactions(U, I, 15000, seed=7)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    return ds


@pytest.fixture(scope='module', params=list(MODELS))
def model(request, train):
    m = MODELS[request.param]()
    m.fit(train, epochs=3, batch_size=64)
    return m


def reference(m, users, items, skip_errors=True):
    """predict() for every pair (distinct pairs once: predict() is deterministic)."""
    memo = {}
    out = []
    for u, i in zip(users.tolist(), items.tolist()):
        if (u, i) not in memo:
            memo[(u, i)] = m.predict(u, i, skip_errors=skip_errors)
        out.append(memo[(u, i)])
    return out


def assert_bitwise(got, want):
    vals = [w for w in want if w is not None]
    assert len(got) == len(want)
    if vals:
        assert {type(w) for w in vals} == {got.dtype.type}, (got.dtype, {type(w) for w in vals})
    for r, w in enumerate(want):
        if w is None:
            assert np.isnan(got[r])
    known = np.array([w is not None for w in want], bool)
    if known.any():
        ref = np.array(vals, got.dtype)
        bits = np.uint32 if got.dtype.itemsize == 4 else np.uint64
        mism = np.flatnonzero(got[known].view(bits) != ref.view(bits))
        assert len(mism) == 0, f'{len(mism)} of {known.sum()} differ, first {got[known][mism[:3]]} vs {ref[mism[:3]]}'


def _random_pairs(train, n, seed):
    rng = np.random.default_rng(seed)
    return (train.raw_users[rng.integers(0, len(train.raw_users), n)],
            train.raw_items[rng.integers(0, len(train.raw_items), n)])


def test_random_pairs_with_duplicates(model, train):
    users, items = _random_pairs(train, 4000, 1)
    assert len(np.unique(users)) > model._max_batch                 # several blocks of users
    got = model.predict_batch(users, items)
    assert_bitwise(got, reference(model, users, items))
    # several device calls: the same values
    assert np.array_equal(model.predict_batch(users, items, chunk=777), got, equal_nan=True)


def test_one_user_with_thousands_of_pairs(model, train):
    rng = np.random.default_rng(2)
    items = train.raw_items[rng.integers(0, len(train.raw_items), 5000)]
    users = np.full(len(items), train.raw_users[17])
    assert_bitwise(model.predict_batch(users, items), reference(model, users, items))


def test_empty_input(model):
    got = model.predict_batch(np.zeros(0, np.int64), np.zeros(0, np.int64))
    assert got.shape == (0,)
    users, items = np.array([model._data.raw_users[0]]), np.array([model._data.raw_items[0]])
    assert got.dtype == model.predict_batch(users, items).dtype


def test_unknown_users_and_items(model, train):
    users, items = _random_pairs(train, 600, 3)
    users[::7] = 10 ** 6                                              # unknown user
    items[3::11] = 10 ** 6 + 1                                        # unknown item
    got = model.predict_batch(users, items, skip_errors=True)
    want = reference(model, users, items)
    assert sum(w is None for w in want) > 50
    assert_bitwise(got, want)
    with pytest.raises(AssertionError, match=f'^User {10 ** 6} was not found.$'):
        model.predict_batch(users, items)
    with pytest.raises(AssertionError, match=f'^Item {10 ** 6 + 1} was not found.$'):
        model.predict_batch(users[3:], items[3:])
    with pytest.raises(AssertionError, match=f'^Item {10 ** 6 + 1} was not found.$'):
        model.predict(users[3], items[3])


def test_after_training_revert_and_reload(train, tmp_path):
    users, items = _random_pairs(train, 2500, 4)
    for name in ('cdae50', 'dmf16_8', 'dmf3'):
        m = MODELS[name]()
        m.fit(train, epochs=3, batch_size=64)
        before = m.predict_batch(users, items)
        m._store_epoch_weights(3)
        for s in range(4, 8):                                         # further training steps
            m._step = s
            m._train_step(64, 1e-3, want_loss=(s == 7))
        after = m.predict_batch(users, items)
        assert not np.array_equal(before, after)
        assert_bitwise(after, reference(m, users, items))
        m._revert_weights(3)                                          # weights written from Python
        assert np.array_equal(m.predict_batch(users, items).view(np.uint8), before.view(np.uint8))
        assert_bitwise(m.predict_batch(users, items), reference(m, users, items))
        path = str(tmp_path / f'{name}.joblib')
        m.save(path)
        m2 = type(m).load(path)
        got = m2.predict_batch(users, items)
        assert np.array_equal(got.view(np.uint8), before.view(np.uint8))
        assert_bitwise(got, reference(m2, users, items))


def test_native_argument_checks(train):
    import torch
    m = MODELS['cdae32']()
    m.fit(train, epochs=1, batch_size=64)
    d = MODELS['dmf16_8']()
    d.fit(train, epochs=1, batch_size=64)
    dev = m._dev

    def t(x, dt):
        return torch.tensor(x, dtype=dt, device=dev)
    ok = dict(users=t([0, 5], torch.int32), off=t([0, 2, 3], torch.int64), iid=t([1, 2, 3], torch.int32),
              dst=t([2, 0, 1], torch.int32))
    bad = [(dict(users=t([0, U], torch.int32)), 'user id'), (dict(users=t([-1, 3], torch.int32)), 'user id'),
           (dict(off=t([0, 3, 2], torch.int64)), 'pair_off'), (dict(off=t([1, 2, 3], torch.int64)), 'pair_off'),
           (dict(off=t([0, 1, 2], torch.int64)), 'pair_off'), (dict(iid=t([1, I, 3], torch.int32)), 'item id'),
           (dict(dst=t([0, 3, 1], torch.int32)), 'output position')]
    P = _lib.t_ptr
    for mdl, fn in ((m, _lib.load().drb_cdae_predict_pairs), (d, _lib.load().drb_dmf_predict_pairs)):
        out = torch.empty(3, dtype=torch.float32, device=dev)
        a = ok
        _lib.check(fn(mdl._native, P(a['users']), 2, P(a['off']), P(a['iid']), P(a['dst']), 3, P(out)))
        for change, msg in bad:
            a = dict(ok, **change)
            with pytest.raises(RuntimeError, match=msg):
                _lib.check(fn(mdl._native, P(a['users']), 2, P(a['off']), P(a['iid']), P(a['dst']), 3, P(out)))
        with pytest.raises(RuntimeError, match='NULL'):
            _lib.check(fn(mdl._native, P(ok['users']), 2, P(ok['off']), None, P(ok['dst']), 3, P(out)))
        with pytest.raises(RuntimeError, match='n_users'):
            _lib.check(fn(mdl._native, P(ok['users']), -1, P(ok['off']), P(ok['iid']), P(ok['dst']), 3, P(out)))
        _lib.check(fn(mdl._native, None, 0, None, None, None, 0, None))      # nothing to do
        # the model still works after the rejected calls
        users, items = _random_pairs(train, 300, 5)
        assert_bitwise(mdl.predict_batch(users, items), reference(mdl, users, items))


def test_item_sharded_cdae_refuses(train):
    m = MODELS['cdae32']()
    m.fit(train, epochs=1, batch_size=64)
    m._sharded = True
    with pytest.raises(NotImplementedError, match='item-sharded'):
        m.predict_batch(train.raw_users[:3], train.raw_items[:3])


@pytest.fixture(scope='module')
def ml20m():
    u, i, v = drb.synthetic_interactions(138493, 26744, 20_000_000, seed=10, zipf_a=1.0)
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=0.2, seed=10, max_concurrent_threads=16)
    train.assign_internal_ids()
    return train, test


@pytest.mark.parametrize('which', ['cdae', 'dmf'])
def test_full_size(ml20m, which):
    train, test = ml20m
    assert len(test) > 3_500_000
    if which == 'cdae':
        m = drb.CDAE(hidden_factors=200, seed=10, verbose=False, rng_mode='philox')
    else:
        m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
    m.fit(train, epochs=2, batch_size=4096)
    got = m.predict_batch(test.user, test.item, skip_errors=True)
    assert len(got) == len(test)
    sample = np.random.default_rng(0).choice(len(test), 2000, replace=False)
    assert_bitwise(got[sample], reference(m, test.user[sample], test.item[sample]))
