"""Host-side pieces of libdrb (no GPU needed): library loads and exports every symbol of include/drb.h, the
CPython RNG replay, PointSampler vs the live-reference goldens, corruption mask vs the oracle, and the
ranking_evaluation protocol vs the live-reference goldens."""
import json
import os
import random
import re
import subprocess
import sys

import numpy as np
import pytest

import drecpy_b200 as drb
from drecpy_b200 import _lib
from oracle.cdae import corruption_keep_mt
from oracle.sampler import PointSamplerOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, 'include', 'drb.h')).read()
    declared = set(re.findall(r'\b(drb_[a-z0-9_]+)\s*\(', header))
    assert declared, 'no declarations parsed'
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in drb.h but not exported'
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.drb_version() == 100


NO_DEVICE_CHILD = '''
import ctypes as C
import torch
import drecpy_b200 as drb
from drecpy_b200 import _lib
assert not torch.cuda.is_available()
h = _lib.vp()
assert _lib.load().drb_ctx_create(0, C.byref(h)) == -2
assert b'no CPU fallback' in _lib.load().drb_last_error()
u, i, v = drb.synthetic_interactions(30, 40, 300)
try:
    drb.CDAE(hidden_factors=8, verbose=False, seed=1).fit(drb.InteractionData(u, i, v), epochs=1)
except RuntimeError:
    pass
else:
    raise AssertionError('fit() ran without a CUDA device')
'''


def test_no_cpu_fallback_without_device():
    """In a child process that sees no CUDA device (so it also runs where a GPU is present)."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, '-c', NO_DEVICE_CHILD], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize('seed', [0, 10, 23, 2 ** 31 + 7, 2 ** 45 + 3])
def test_rng_replays_cpython(seed):
    lib = _lib.load()
    g = _lib.HostRng(seed)
    r = random.Random(seed)
    assert [g.random() for _ in range(1500)] == [r.random() for _ in range(1500)]
    for n in [1, 2, 3, 7, 943, 1682, 10 ** 6, 2 ** 32, 2 ** 40 + 11]:
        assert [g.randbelow(n) for _ in range(40)] == [r._randbelow(n) for _ in range(40)]
    for k in [1, 7, 31, 32, 33, 53, 64]:
        assert lib.drb_rng_getrandbits(g.handle, k) == r.getrandbits(k)
    st = r.getstate()[1]
    assert np.array_equal(g.getstate(), np.array(st, np.uint32))
    # sample / shuffle (CPython 3.12 algorithms)
    for n, k in [(5, 3), (21, 6), (100, 7), (101, 100), (1000, 100), (4000, 21), (30, 0)]:
        out = np.zeros(max(k, 1), np.int64)
        _lib.check(lib.drb_rng_sample_indices(g.handle, n, k, _lib.np_ptr(out)))
        assert out[:k].tolist() == r.sample(range(n), k), (n, k)
    x = np.arange(101, dtype=np.int64)
    y = list(range(101))
    _lib.check(lib.drb_rng_shuffle_i64(g.handle, 101, _lib.np_ptr(x)))
    r.shuffle(y)
    assert x.tolist() == y


@pytest.mark.parametrize('name', ['small_zero_rows', 'small_dups', 'small_float', 'thr3'])
def test_native_sampler_and_csr_vs_live_reference(golden_dir, name):
    g = np.load(os.path.join(golden_dir, f'sampler_{name}.npz'))
    ds = drb.InteractionData(g['user'], g['item'], g['interaction'])
    ds.assign_internal_ids()
    assert np.array_equal(ds.uid, g['uid']) and np.array_equal(ds.iid, g['iid'])
    for got, want in zip(ds.csr(), (g['csr_indptr'], g['csr_indices'], g['csr_data'])):
        assert np.array_equal(got, want)
    for got, want in zip(ds.csc(), (g['csc_indptr'], g['csc_indices'], g['csc_data'])):
        assert np.array_equal(got, want)
    assert np.array_equal(ds.select_user_interaction_vec(0).toarray().ravel(), g['dense_user0'])
    assert np.array_equal(ds.select_item_interaction_vec(0).toarray().ravel(), g['dense_item0'])
    for key in g.files:
        if key.startswith('triples_seed'):
            seed = int(key[len('triples_seed'):])
            s = drb.PointSampler(ds, int(g['neg_ratio']), float(g['thr']), seed)
            u, i, v = s.sample_arrays(len(g[key]))
            assert np.array_equal(np.stack([u, i, v], 1).astype(np.float64), g[key]), (name, seed)


def test_native_sampler_vs_oracle_c1_shape_and_state_roundtrip():
    u, i, v = drb.synthetic_interactions(943, 1682, 100000, seed=10)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    assert ds.count_unique('uid') == 943 and ds.count_unique('iid') == 1682
    s = drb.PointSampler(ds, 5, 0.001, 10)
    o = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 0.001, 10)
    assert s.sample(640) == [(a, b, int(c)) for a, b, c in o.sample(640)]
    st = s.getstate()
    a = s.sample(50)
    s.setstate(st)
    assert s.sample(50) == a


@pytest.mark.parametrize('density,neg_ratio', [(0.9, 5), (0.5, 1), (0.02, 9)])
def test_native_sampler_stream_decoupling_under_heavy_rejection(density, neg_ratio):
    """The native sampler walks the reference's three independent random.Random streams one after the other (decisions,
    null pairs in blocks no longer than the number of open samples, positives) instead of sample by sample.  With a
    nearly full matrix most null candidates are stored pairs and get skipped, with users without positives the
    positive generator redraws: outputs, call boundaries (1, 7, 300 samples per call) and the final states of all
    three streams must still equal the sample-by-sample oracle."""
    rng = np.random.default_rng(3)
    U, I = 60, 45
    mask = rng.random((U, I)) < density
    mask[7] = False                                           # a user without any interaction
    uu, ii = np.nonzero(mask)
    vv = rng.integers(0, 3, len(uu))                          # zeros: stored rows below the threshold
    keep = np.ones(len(uu), bool)
    ds = drb.InteractionData(uu[keep], ii[keep], vv[keep])
    ds.assign_internal_ids()
    s = drb.PointSampler(ds, neg_ratio, 1, 10)
    o = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, neg_ratio, 1, 10)
    for n in (1, 7, 300, 0, 2):
        got = s.sample(n)
        want = [(a, b, int(c)) for a, b, c in o.sample(n)] if n else []
        assert got == want, n
    # one more draw from every stream: the states agree, not only the outputs so far
    assert s.sample(64) == [(a, b, int(c)) for a, b, c in o.sample(64)]


def test_corruption_mask_matches_python_stream():
    """cdae.py:63-64: n_items draws per sampled user, in item order; the native replay skips unused draws."""
    u, i, v = drb.synthetic_interactions(60, 97, 900, seed=3)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    indptr, indices, _ = ds.csr(0.001)
    uids = np.array([5, 17, 5, 0, 59, 33], np.int32)
    rng = _lib.HostRng(10)
    off = np.zeros(len(uids) + 1, np.int32)
    keep = np.zeros(int(np.diff(indptr).max()) * len(uids), np.uint8)
    _lib.check(_lib.load().drb_cdae_corruption_keep_mt(rng.handle, _lib.np_ptr(uids), len(uids), 97, 0.2,
                                                       _lib.np_ptr(indptr), _lib.np_ptr(indices), _lib.np_ptr(off),
                                                       _lib.np_ptr(keep), len(keep)))
    pr = random.Random(10)
    for b, uid in enumerate(uids):
        dense = corruption_keep_mt(pr, 97, 0.2)
        items = indices[indptr[uid]:indptr[uid + 1]]
        assert np.array_equal(keep[off[b]:off[b + 1]].astype(bool), dense[items])
    assert rng.random() == pr.random()          # both streams consumed exactly len(uids) * n_items draws


def test_corruption_mask_refuses_a_short_keep_buffer():
    """Users repeat inside a batch (sampling is with replacement), so batch nnz is not bounded by any set of distinct
    users: the native replay takes the buffer capacity, fails without writing and without consuming draws."""
    u, i, v = drb.synthetic_interactions(20, 50, 400, seed=3)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    indptr, indices, _ = ds.csr(0.001)
    heavy = int(np.argmax(np.diff(indptr)))
    uids = np.full(64, heavy, np.int32)                      # batch_size > n_users, one user repeated
    nnz = int(np.diff(indptr)[heavy]) * len(uids)
    assert nnz > int(np.diff(indptr).sum())                  # more than the whole dataset holds
    rng = _lib.HostRng(10)
    off = np.zeros(len(uids) + 1, np.int32)
    guard = np.full(nnz + 64, 0xAB, np.uint8)
    rc = _lib.load().drb_cdae_corruption_keep_mt(rng.handle, _lib.np_ptr(uids), len(uids), 50, 0.2,
                                                 _lib.np_ptr(indptr), _lib.np_ptr(indices), _lib.np_ptr(off),
                                                 _lib.np_ptr(guard), nnz - 1)
    assert rc == -1 and b'room for' in _lib.load().drb_last_error()
    assert (guard == 0xAB).all() and rng.random() == random.Random(10).random()
    rng = _lib.HostRng(10)
    _lib.check(_lib.load().drb_cdae_corruption_keep_mt(rng.handle, _lib.np_ptr(uids), len(uids), 50, 0.2,
                                                       _lib.np_ptr(indptr), _lib.np_ptr(indices), _lib.np_ptr(off),
                                                       _lib.np_ptr(guard), nnz))
    assert off[-1] == nnz and (guard[nnz:] == 0xAB).all() and set(np.unique(guard[:nnz])) <= {0, 1}


class FakeModel:
    def __init__(self, train):
        self.interaction_dataset = self._data = train
        self.interaction_threshold = 0.001
        self.n_items = train.count_unique('iid')

    def rank(self, user, items, novelty=True, skip_invalid_items=True, **kw):
        t = self._data
        uid = t.user_to_uid(user)
        cand = set(x for x in (t.item_to_iid(it) for it in items) if x is not None)
        if novelty:
            cand -= set(t.user_items(uid).tolist())
        r = sorted([(float((uid * 7919 + i * 104729) % 97) / 97.0, i) for i in cand], reverse=True)
        return [(s, t.iid_to_item(i)) for s, i in r]


def test_ranking_evaluation_protocol_vs_live_reference(golden_dir):
    with open(os.path.join(golden_dir, 'ranking.json')) as f:
        g = json.load(f)
    tr, te = np.array(g['train_rows']), np.array(g['test_rows'])
    train = drb.InteractionData(*[tr[:, c].astype(np.int64) for c in range(3)])
    train.assign_internal_ids()
    test = drb.InteractionData(*[te[:, c].astype(np.int64) for c in range(3)])
    for name, case in g['cases'].items():
        rec = []
        res = drb.ranking_evaluation(FakeModel(train), test, record=rec, **case['kwargs'])
        assert res == case['result'], name
        assert len(rec) == len(case['per_user'])
        for user, cands, ranked in rec:
            ref = case['per_user'][str(user)]
            assert cands == ref['candidates'] and ranked == ref['ranked'], (name, user)


def test_ranking_evaluation_argument_errors():
    """error behaviour of ranking_evaluation.py:63-71 (reference tests test_ranking_evaluation.py:127-250)."""
    u, i, v = drb.synthetic_interactions(20, 30, 200)
    train = drb.InteractionData(u, i, v)
    train.assign_internal_ids()
    m = FakeModel(train)
    with pytest.raises(AssertionError, match=r'The number of test users \(0\) should be > 0.'):
        drb.ranking_evaluation(m, train, n_test_users=0)
    with pytest.raises(AssertionError, match=r'k \(0\) should be > 0.'):
        drb.ranking_evaluation(m, train, k=0)
    with pytest.raises(Exception, match='Cannot generate negative interaction pairs'):
        drb.ranking_evaluation(m, train, generate_negative_pairs=True)
    with pytest.raises(AssertionError, match='Expected "metrics" argument to be a list'):
        drb.ranking_evaluation(m, train, metrics=drb.NDCG())


class FakeBatchModel(FakeModel):
    """FakeModel plus the batched rank_arrays() entry the vectorised evaluator uses."""

    def rank_arrays(self, user_ids, cand, cand_off, novelty=True, chunk=0):
        n = len(user_ids)
        c_max = int(np.diff(cand_off).max())
        out = np.full((n, c_max), -1, np.int64)
        n_out = np.zeros(n, np.int32)
        for r, user in enumerate(np.asarray(user_ids).tolist()):
            ranked = [it for _, it in self.rank(user, cand[cand_off[r]:cand_off[r + 1]].tolist(), novelty=novelty)]
            out[r, :len(ranked)] = ranked
            n_out[r] = len(ranked)
        return out, n_out


def test_vectorised_evaluation_equals_per_user_protocol(golden_dir):
    with open(os.path.join(golden_dir, 'ranking.json')) as f:
        g = json.load(f)
    tr, te = np.array(g['train_rows']), np.array(g['test_rows'])
    train = drb.InteractionData(*[tr[:, c].astype(np.int64) for c in range(3)])
    train.assign_internal_ids()
    test = drb.InteractionData(*[te[:, c].astype(np.int64) for c in range(3)])
    model = FakeBatchModel(train)
    for name, case in g['cases'].items():
        fast = drb.ranking_evaluation(model, test, **case['kwargs'])
        assert fast == case['result'], name                       # the live reference's own result
    # random protocol settings on a bigger synthetic split: fast path == general path
    u, i, v = drb.synthetic_interactions(300, 400, 9000, seed=21)
    v = v - 1                                                     # include zero-valued (sub-threshold) rows
    rng = np.random.default_rng(5)
    mask = rng.random(len(u)) < 0.2
    train = drb.InteractionData(u[~mask], i[~mask], v[~mask])
    train.assign_internal_ids()
    test = drb.InteractionData(u[mask], i[mask], v[mask])
    model = FakeBatchModel(train)
    for kw in [dict(k=[1, 5, 10], n_pos_interactions=1, n_neg_interactions=100, generate_negative_pairs=True,
                    novelty=True, seed=10),
               dict(k=3, n_pos_interactions=None, n_neg_interactions=None, novelty=False),
               dict(k=[2, 7], n_pos_interactions=2, n_neg_interactions=0.5, generate_negative_pairs=True, seed=4),
               dict(k=10, n_pos_interactions=None, n_neg_interactions=5, novelty=True, n_test_users=50)]:
        fast = drb.ranking_evaluation(model, test, verbose=False, **kw)
        slow = drb.ranking_evaluation(model, test, verbose=False, force_python=True, **kw)
        assert fast == slow, (kw, fast, slow)


def test_vectorised_evaluation_with_duplicate_test_rows_and_ragged_lists():
    """The vectorised evaluator checks the users' TEST ROWS for repeated items first (a candidate list can only repeat an
    item when they do) and only then the lists themselves; with duplicates it must hand over to the general path, and
    without generated negatives the lists are ragged (segment arithmetic instead of a reshape)."""
    u, i, v = drb.synthetic_interactions(200, 300, 6000, seed=33)
    rng = np.random.default_rng(8)
    mask = rng.random(len(u)) < 0.25
    train = drb.InteractionData(u[~mask], i[~mask], v[~mask])
    train.assign_internal_ids()
    tu, ti, tv = u[mask], i[mask], v[mask]
    dup = rng.choice(len(tu), 40, replace=False)                  # repeat 40 test rows: same (user, item) twice
    test_dup = drb.InteractionData(np.concatenate([tu, tu[dup]]), np.concatenate([ti, ti[dup]]),
                                   np.concatenate([tv, tv[dup]]))
    test_plain = drb.InteractionData(tu, ti, tv)
    model = FakeBatchModel(train)
    for test in (test_dup, test_plain):
        for kw in [dict(k=[3, 10], n_pos_interactions=None, n_neg_interactions=None, novelty=False),            # ragged
                   dict(k=5, n_pos_interactions=1, n_neg_interactions=50, generate_negative_pairs=True, seed=3),  # uniform
                   dict(k=[1, 4], n_pos_interactions=None, n_neg_interactions=7, novelty=True, seed=6)]:
            fast = drb.ranking_evaluation(model, test, verbose=False, **kw)
            slow = drb.ranking_evaluation(model, test, verbose=False, force_python=True, **kw)
            assert fast == slow, (kw, fast, slow)


def test_native_metric_sums_equal_the_metric_classes():
    """drb_eval_metrics against the metric classes (restated from Evaluation/Metrics/ranking.py:20-114) user by user:
    short and long test tables (linear scan / sorted index), few and many positives, real-valued relevancies with
    repeated test rows (first row wins), ranked lists shorter than k, cut-offs beyond the list length."""
    import ctypes as C
    from drecpy_b200 import _lib
    rng = np.random.default_rng(12)
    n, L, ks = 40, 30, [1, 3, 10, 50]
    t_beg, t_end, t_key, t_val, c_beg, c_end, c_key, p_beg, p_end, p_key = [], [], [], [], [], [], [], [], [], []
    ranked = np.full((n, L), -1, np.int64)
    n_out = np.zeros(n, np.int32)
    for g in range(n):
        nt = int(rng.integers(0, 40))                              # test rows of the user (some > 16: sorted path)
        keys = rng.integers(0, 60, nt)
        t_beg.append(len(t_key)); t_key += keys.tolist(); t_val += rng.choice([0.0, 1.0, 2.5, 4.0], nt).tolist()
        t_end.append(len(t_key))
        cands = rng.permutation(80)[:int(rng.integers(1, L + 1))]
        c_beg.append(len(c_key)); c_key += cands.tolist(); c_end.append(len(c_key))
        pos = rng.permutation(cands)[:int(rng.integers(1, min(len(cands), 25) + 1))]
        p_beg.append(len(p_key)); p_key += pos.tolist(); p_end.append(len(p_key))
        r = rng.permutation(cands)[:int(rng.integers(0, len(cands) + 1))]     # the model may drop candidates (novelty)
        ranked[g, :len(r)] = r; n_out[g] = len(r)
    arr = lambda x, t: np.ascontiguousarray(x, t)
    A = dict(t_beg=arr(t_beg, np.int64), t_end=arr(t_end, np.int64), t_key=arr(t_key, np.int64), t_val=arr(t_val, np.float64),
             c_beg=arr(c_beg, np.int64), c_end=arr(c_end, np.int64), c_key=arr(c_key, np.int64),
             p_beg=arr(p_beg, np.int64), p_end=arr(p_end, np.int64), p_key=arr(p_key, np.int64), ks=arr(ks, np.int64))
    dcg, idcg = np.zeros((n, len(ks))), np.zeros((n, len(ks)))
    hits = np.zeros((n, len(ks)), np.int64)
    P = _lib.np_ptr
    _lib.check(_lib.load().drb_eval_metrics(n, P(A['t_beg']), P(A['t_end']), P(A['t_key']), P(A['t_val']), P(ranked), L,
                                            P(n_out), P(A['c_beg']), P(A['c_end']), P(A['c_key']), P(A['p_beg']),
                                            P(A['p_end']), P(A['p_key']), P(A['ks']), len(ks), 1, P(dcg), P(idcg), P(hits)))
    ndcg, dcg_m, hr, prec = drb.NDCG(), drb.DCG(), drb.HitRatio(), drb.Precision()
    for g in range(n):
        rel = {}
        for it in c_key[c_beg[g]:c_end[g]]:
            first = [t_val[r] for r in range(t_beg[g], t_end[g]) if t_key[r] == it]
            rel[it] = first[0] if first else 0
        rec = ranked[g, :n_out[g]].tolist()
        positives = p_key[p_beg[g]:p_end[g]]
        for j, k in enumerate(ks):
            assert dcg[g, j] == dcg_m(rec, k=k, relevancies=rel), (g, k)
            best = sorted(rel, key=lambda x: -rel[x])
            assert idcg[g, j] == dcg_m(best, k=k, relevancies=rel), (g, k)
            if idcg[g, j] != 0:
                assert dcg[g, j] / idcg[g, j] == ndcg(rec, k=k, relevancies=rel)
            assert hits[g, j] / len(positives) == hr(rec, k=k, relevant_recommendations=positives)
            if min(k, len(rec)):
                assert hits[g, j] / min(k, len(rec)) == prec(rec, k=k, relevant_recommendations=positives)


# ------------------------------------------------------------------------------------------------ leave_k_out
def test_leave_k_out_matches_live_reference_goldens():
    """drecpy_b200.leave_k_out (native per-user Random(seed + idx + 1).sample replay) against the row ids the live
    reference produced (tests/golden/splits.json <- DRecPy/Evaluation/Splits/leave_k_out.py:14-135): fixed and ratio
    k, min_user_interactions, k above some users' history length, last_timestamps."""
    import json
    g = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'splits.json')))
    rows = np.array(g['rows'], dtype=np.int64)
    ds = drb.InteractionData(rows[:, 0], rows[:, 1], rows[:, 2])
    key = {(int(u), int(i)): r for r, (u, i) in enumerate(zip(rows[:, 0], rows[:, 1]))}    # (user, item) pairs are unique
    for name, case in g['cases'].items():
        kw = dict(case['kwargs'])
        train, test = drb.leave_k_out(ds, timestamps=rows[:, 3], verbose=False, **kw)
        tr = [key[(int(u), int(i))] for u, i in zip(train.user, train.item)]
        te = [key[(int(u), int(i))] for u, i in zip(test.user, test.item)]
        assert tr == sorted(tr) and te == sorted(te), name              # input row order is preserved
        assert tr == case['train_rid'], name
        assert te == case['test_rid'], name


def test_leave_k_out_reference_fixture_and_errors():
    """The reference's own evaluation fixture (tests/Evaluation/Processes/test_ranking_evaluation.py:12-19): the split
    stored in ranking.json came from the live leave_k_out(k=5, seed=10)."""
    import json, random
    g = json.load(open(os.path.join(os.path.dirname(__file__), 'golden', 'ranking.json')))
    rng = random.Random(0)
    rows = np.array([[u, i, rng.randint(-1, 5)] for u in range(50) for i in range(200) if rng.randint(0, 4) == 0])
    train, test = drb.leave_k_out(drb.InteractionData(rows[:, 0], rows[:, 1], rows[:, 2]), k=5, seed=10, verbose=False)
    assert np.stack([train.user, train.item, train.interaction], 1).tolist() == g['train_rows']
    assert np.stack([test.user, test.item, test.interaction], 1).tolist() == g['test_rows']
    # multi-threaded path (>= 1024 users) equals the single-threaded one: users are independent
    rs = np.random.default_rng(0)
    u = np.repeat(np.arange(3000), 12); i = rs.integers(0, 10**6, len(u)); v = np.ones(len(u), np.int64)
    a = drb.leave_k_out(drb.InteractionData(u, i, v), k=2, seed=4, max_concurrent_threads=8, verbose=False)
    b = drb.leave_k_out(drb.InteractionData(u, i, v), k=2, seed=4, max_concurrent_threads=1, verbose=False)
    assert np.array_equal(a[1].item, b[1].item) and len(a[1]) == 6000 and len(a[0]) == 30000
    with pytest.raises(AssertionError):
        drb.leave_k_out(drb.InteractionData(u, i, v), k=0)
    with pytest.raises(Exception, match='should be in the'):
        drb.leave_k_out(drb.InteractionData(u, i, v), k=1.5)


# ------------------------------------------------------------------------------------------------ repo contracts
def test_product_package_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under drecpy_b200/ may import or execute it."""
    root = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'drecpy_b200')
    for name in os.listdir(root):
        if name.endswith('.py'):
            src = open(os.path.join(root, name)).read()
            assert not re.search(r'^\s*(from|import)\s+oracle\b', src, re.M), name


def test_committed_bench_lines_carry_the_contract_keys():
    """profiles/r1_bench_n*.json are bench.py's own output lines: every key the bench contract names is present."""
    prof = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles')
    for n in (1, 2, 4, 8):
        j = json.load(open(os.path.join(prof, f'r1_bench_n{n}.json')))
        for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                  'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'gpu_launches', 'e2e', 'roofline'):
            assert k in j, (n, k)
        assert j['n_gpus'] == n and j['warmup'] >= 3 and j['vs_baseline'] is None and 'workload' in j['config']
        assert set(j['e2e']) >= {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
        assert set(j['roofline']) >= {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'}
        assert j['gpu_launches'] > 0 and j['e2e']['value'] < j['value']
        assert not set(j['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
        if n == 1:
            assert set(j['cpu_baseline']) >= {'value', 'unit', 'cores', 'kind', 'sample'}
            assert abs(j['roofline']['frac'] - j['roofline']['achieved'] / j['roofline']['peak']) < 1e-9


def test_rank_arrays_uniform_and_ragged_paths_agree():
    """DeepRecommenderABC.rank_arrays (host side of the batched scorer): the reshape fast path for equally long
    candidate lists and the padded path for ragged ones hand the same lists to _rank_batch and map the same raw ids
    back, including unknown items (-1) and rows shortened by the novelty filter."""
    from drecpy_b200.recommender import DeepRecommenderABC

    class Scorer(DeepRecommenderABC):
        def __init__(self, data):
            self._data = data
            self.n_items = data.count_unique('iid')

        def _pre_fit(self, *a, **k): pass
        def _predict(self, *a, **k): pass
        def _train_step(self, *a, **k): pass

        def _rank_batch(self, uids, cand, cand_count, novelty):
            n, c = cand.shape
            oi, on = np.full((n, c), -1, np.int32), np.zeros(n, np.int32)
            for r in range(n):
                items = [int(x) for x in cand[r, :cand_count[r]] if x >= 0]
                if novelty:
                    seen = set(self._data.user_items(int(uids[r])).tolist())
                    items = [x for x in items if x not in seen]
                items = sorted(set(items), key=lambda x: ((x * 2654435761 + int(uids[r])) % 1009, x), reverse=True)
                oi[r, :len(items)] = items
                on[r] = len(items)
            return oi, np.zeros((n, c), np.float32), on

    u, i, v = drb.synthetic_interactions(40, 60, 600, seed=2)
    data = drb.InteractionData(u, i, v)
    data.assign_internal_ids()
    m = Scorer(data)
    rng = np.random.default_rng(1)
    users = data.raw_users[rng.permutation(40)[:25]]
    for novelty in (False, True):
        uniform = rng.integers(1, 61, (25, 12)).astype(np.int64)
        uniform[3, 5] = 10_000                                       # unknown raw item
        off = np.arange(26, dtype=np.int64) * 12
        got, n_out = m.rank_arrays(users, uniform.reshape(-1), off, novelty=novelty, chunk=7)
        # the same lists, made ragged by appending one extra list of a different length
        cand2 = np.concatenate([uniform.reshape(-1), np.array([5, 6, 7], np.int64)])
        off2 = np.concatenate([off, [off[-1] + 3]])
        got2, n_out2 = m.rank_arrays(np.concatenate([users, users[:1]]), cand2, off2, novelty=novelty, chunk=7)
        assert np.array_equal(n_out, n_out2[:25]) and np.array_equal(got, got2[:25, :12])
        for r in range(25):
            uid = data.user_to_uid(users[r].item())
            iids = [data.item_to_iid(int(x)) for x in uniform[r]]
            iids = [x for x in iids if x is not None]
            if novelty:
                iids = [x for x in iids if x not in set(data.user_items(uid).tolist())]
            exp = sorted(set(iids), key=lambda x: ((x * 2654435761 + uid) % 1009, x), reverse=True)
            assert got[r, :n_out[r]].tolist() == [data.iid_to_item(x) for x in exp]
            assert (got[r, n_out[r]:] == -1).all()


def test_config4_flow_split_then_evaluate_small():
    """Config 4's host flow end to end at a small shape: leave_k_out(k=1) -> ranking_evaluation with 1 positive and
    generated negatives; the vectorised evaluator (native candidates + grouped lookups) equals the per-user protocol."""
    u, i, v = drb.synthetic_interactions(250, 320, 7000, seed=9)
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=1, seed=10, verbose=False)
    assert len(test) == 250 and len(train) == 7000 - 250
    train.assign_internal_ids()
    model = FakeBatchModel(train)
    kw = dict(k=[5, 10], n_pos_interactions=1, n_neg_interactions=100, generate_negative_pairs=True, novelty=True,
              seed=10, metrics=[drb.HitRatio(), drb.NDCG(), drb.Precision(), drb.Recall()])
    fast = drb.ranking_evaluation(model, test, verbose=False, **kw)
    slow = drb.ranking_evaluation(model, test, verbose=False, force_python=True, **kw)
    assert fast == slow and 0 < fast['HitRatio@10'] <= 1


def test_bench_roofline_object_from_committed_kernel_times():
    """bench.cdae_roofline is the pure part of the bench line: fed with the kernel times of the committed round-1 one-GPU
    line and the committed ncu traffic table it reproduces that line's roofline numbers."""
    import importlib.util
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location('bench_module', os.path.join(root, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    j = json.load(open(os.path.join(root, 'profiles', 'r1_bench_n1.json')))
    table = json.load(open(os.path.join(root, 'profiles', 'r1_traffic.json')))['dram_bytes_per_launch']
    peaks = dict(hbm=j['roofline']['secondary']['k_adam']['peak'], tf=j['roofline']['peak'], tf_burst=0.0, src='measured')
    n_params = 2 * 26744 * 200 + 138493 * 200 + 200 + 26744                 # W, W', V, b, b' (ld == hidden == 200)
    r = bench.cdae_roofline(j['kernels_ms_per_step'], bench.C3, n_params, peaks, table)
    assert r['bound'] == 'tensor' and r['unit'] == 'TFLOP/s'
    assert abs(r['achieved'] - j['roofline']['achieved']) < 1e-6 * r['achieved']
    assert abs(r['frac'] - r['achieved'] / r['peak']) < 1e-12
    assert r['traffic'] == table['k_umma_cdae_loss'] + table['k_umma_gemm_mn'] + table['k_umma_gemm_kk']
    assert abs(r['algorithmic_flops_per_step'] - 6.0 * 200 * 26744 * 4096) < 1
    assert 0.8 < r['secondary']['k_adam']['frac'] < 1.0
    # the closing round-2 line with the newest committed traffic table (what bench.py itself loads)
    j2 = json.loads(open(os.path.join(root, 'profiles', 'r2_bench_n1.json')).read().strip().splitlines()[-1])
    t2 = bench.load_traffic()
    assert {'k_umma_cdae_loss', 'k_umma_gemm_dw', 'k_umma_gemm_dh', 'k_adam'} <= set(t2)
    r3 = bench.cdae_roofline(j2['kernels_ms_per_step'], bench.C3, n_params, peaks, t2)
    assert abs(r3['frac'] - j2['roofline']['frac']) < 1e-9 and 0.2 < r3['frac'] < 0.3
    assert r3['traffic'] == t2['k_umma_cdae_loss'] + t2['k_umma_gemm_dw'] + t2['k_umma_gemm_dh'] < 1.6e9
    # Adam: 28 B per parameter minus the unread gradient of user rows without a sampled user (N ranks touch N batches)
    a1 = r3['secondary']['k_adam']['algorithmic_bytes_per_step']
    a8 = bench.cdae_roofline(j2['kernels_ms_per_step'], bench.C3, n_params, peaks, t2, world=8)['secondary']['k_adam']
    assert a1 == 28.0 * n_params - 4.0 * (138493 - 4096) * 200
    assert a8['algorithmic_bytes_per_step'] == 28.0 * n_params - 4.0 * (138493 - 8 * 4096) * 200
    # FFMA path: no traffic claim
    r2 = bench.cdae_roofline({'k_sgemm_kk_loss': 2.5, 'k_sgemm_mn': 1.7, 'k_sgemm_kn': 2.8, 'k_adam': 0.17}, bench.C3,
                             n_params, peaks, table)
    assert r2['traffic'] is None and r2['achieved'] > 0
    # every workload has a native and a reference runner
    for name, cfg in bench.WORKLOADS.items():
        assert cfg['model'] in bench.RUNNERS and len(bench.RUNNERS[cfg['model']]) == 2, name
