"""DMF full-catalog top-k (drb_dmf_topk, dmf_topk.cu): every row is bit for bit what the rank path
(drb_dmf_rank_candidates over the whole catalog) returns for that user, truncated to k -- the same item ids in the same
order and the same fp32 scores.  Also: against the oracle, exact ties across a pass boundary, the 1e-6 score floor,
users with few unseen items, list overflow, tower widths, the item-tower cache, the public surface and the errors."""
import heapq

import numpy as np
import pytest

import drecpy_b200 as drb
from drecpy_b200 import _lib
from oracle.dmf import DMFOracle

pytestmark = pytest.mark.gpu


def _weights(U, I, uf, itf, seed=2):
    rng = np.random.default_rng(seed)

    def tower(in_dim, factors):
        out = []
        for f in factors:
            lim = np.sqrt(6.0 / (in_dim + f))
            out.append((rng.uniform(-lim, lim, (in_dim, f)).astype(np.float32),
                        rng.uniform(0.0, 0.05, f).astype(np.float32)))
            in_dim = f
        return out
    return {'user_nn': tower(I, uf), 'item_nn': tower(U, itf)}


def _data(U, I, nnz, seed=5, rows=None):
    """Interactions with internal item id == raw item id - 1 (rows sorted by item before the ids are assigned)."""
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=seed)
    if rows is not None:
        u, i, v = rows(u, i, v)
    o = np.argsort(i, kind='stable')
    ds = drb.InteractionData(u[o], i[o], v[o])
    ds.assign_internal_ids()
    return ds


def _model(ds, uf=(64, 32), itf=(64, 32), score_batch=0, w=None):
    uf, itf = list(uf), list(itf)
    w = w or _weights(ds.count_unique('uid'), ds.count_unique('iid'), uf, itf)
    m = drb.DMF(user_factors=uf, item_factors=itf, seed=10, verbose=False)
    m.fit(ds, epochs=0, batch_size=64, init_weights=w, score_batch=score_batch)
    return m, w


def _rank_all(m, uids, novelty):
    """The rank path over the whole catalog: (iids, raw fp32 scores, n_out) host arrays."""
    torch = m._torch
    d_u = torch.as_tensor(np.asarray(uids, np.int32), device=m._dev)
    cat = torch.arange(m.n_items, dtype=torch.int32, device=m._dev)
    out_i, out_s, out_n = [], [], []
    for o in range(0, len(uids), 512):
        c = d_u[o:o + 512].numel()
        oi, os_, on = m._rank_device(d_u[o:o + 512].contiguous(), cat.expand(c, -1).contiguous(),
                                     torch.full((c,), m.n_items, dtype=torch.int32, device=m._dev), novelty)
        out_i.append(oi.cpu().numpy()), out_s.append(os_.cpu().numpy()), out_n.append(on.cpu().numpy())
    return np.concatenate(out_i), np.concatenate(out_s), np.concatenate(out_n)


def _topk_raw(m, uids, k, novelty, scratch_bytes=None):
    """drb_dmf_topk through the C ABI: raw fp32 scores, n_out == -1 left as the library reports it."""
    torch = m._torch
    lib = _lib.load()
    m._sync_item_cache()
    nb = lib.drb_dmf_topk_scratch_bytes(m._native, k)
    scratch = torch.empty(max(nb, 256), dtype=torch.uint8, device=m._dev)
    d_u = torch.as_tensor(np.asarray(uids, np.int32), device=m._dev)
    n = d_u.numel()
    o_i = torch.empty((n, k), dtype=torch.int32, device=m._dev)
    o_s = torch.empty((n, k), dtype=torch.float32, device=m._dev)
    o_n = torch.empty(n, dtype=torch.int32, device=m._dev)
    _lib.check(lib.drb_dmf_topk(m._native, _lib.t_ptr(d_u), n, k, 1 if novelty else 0, _lib.t_ptr(scratch),
                                nb if scratch_bytes is None else scratch_bytes, _lib.t_ptr(o_i), _lib.t_ptr(o_s),
                                _lib.t_ptr(o_n)))
    return o_i.cpu().numpy(), o_s.cpu().numpy(), o_n.cpu().numpy()


def _assert_same(got, ref, k):
    """got = (iids, scores, n_out) of the top-k; ref = the rank path's full lists: equal ids, equal score bits."""
    gi, gs, gn = got
    ri, rs, rn = ref
    np.testing.assert_array_equal(gn, np.minimum(rn, k))
    valid = np.arange(k)[None, :] < gn[:, None]
    np.testing.assert_array_equal(np.where(valid, gi, -1), np.where(valid, ri[:, :k], -1))
    bits = np.uint32 if gs.dtype == np.float32 else np.uint64
    np.testing.assert_array_equal(np.where(valid, gs.view(bits), 0), np.where(valid, rs[:, :k].astype(gs.dtype).view(bits), 0))


def _profile(m, fn):
    lib = _lib.load()
    m.synchronize()
    _lib.check(lib.drb_ctx_profile_enable(m._ctx, 1))
    _lib.profile_read(m._ctx)
    try:
        out = fn()
        m.synchronize()
        return out, _lib.profile_read(m._ctx)
    finally:
        _lib.check(lib.drb_ctx_profile_enable(m._ctx, 0))


@pytest.fixture(scope='module')
def c2():
    ds = _data(6040, 3706, 1_000_000, seed=5)
    m, w = _model(ds)
    return ds, m, w


@pytest.fixture(scope='module')
def wide():
    ds = _data(700, 9000, 60000, seed=6)
    m, w = _model(ds)
    return ds, m, w


# ------------------------------------------------------------------ 1. bitwise equality with the rank path
@pytest.mark.parametrize('shape', ['c2', 'wide'])
@pytest.mark.parametrize('novelty', [True, False])
def test_topk_equals_rank_path_bitwise(shape, novelty, request):
    ds, m, _ = request.getfixturevalue(shape)
    uids = np.arange(m.n_users, dtype=np.int32)
    ref = _rank_all(m, uids, novelty)
    for k in (1, 37, 100, 2048):
        got = _topk_raw(m, uids, k, novelty)
        _assert_same(got, ref, k)
        # the public entry: the same ids, scores rescaled exactly as rank() rescales them
        ti, ts, tn = m.topk_batch(uids, k, novelty)
        _assert_same((ti, ts, tn), (ref[0], m._rescale_value(ref[1]), ref[2]), k)


def test_topk_does_not_depend_on_the_block(wide):
    """Blocks of 1024 users (2500 rows: three blocks, the last one partial) and one block of 4096: uids shuffled and
    repeated, the same answer as the rank path row for row."""
    ds, m, w = wide
    rng = np.random.default_rng(0)
    uids = np.concatenate([rng.permutation(m.n_users)] * 3 + [rng.integers(0, m.n_users, 400)]).astype(np.int32)
    ref = _rank_all(m, uids, True)
    for sb in (1024, 4096):
        mb, _ = _model(ds, score_batch=sb, w=w)
        assert mb._max_batch == sb
        _assert_same(_topk_raw(mb, uids, 100, True), ref, 100)


# ------------------------------------------------------------------ 2. against the oracle
def test_topk_against_oracle(c2):
    ds, m, w = c2
    o = DMFOracle(w['user_nn'], w['item_nn'], ds.csr(), ds.csc(), m.min_interaction, m.max_interaction)
    I = m.n_items
    uids = np.array([0, 17, 999, 3000, 6039], np.int32)
    gi, gs, gn = _topk_raw(m, uids, 100, True)
    near = 0
    for r, uid in enumerate(uids):
        p = o.forward(np.full(I, uid), np.arange(I))[0]
        seen = set(ds.user_items(int(uid)).tolist())
        want = heapq.nlargest(100, ((float(p[i]), i) for i in range(I) if i not in seen))
        assert gn[r] == len(want)
        got = gi[r, :gn[r]].tolist()
        if got != [i for _, i in want]:
            near += 1
            for a, (sb, b) in zip(got, want):
                if a != b:
                    assert abs(p[a] - sb) <= 2e-6 * max(abs(p[a]), abs(sb)), (uid, a, b, p[a], sb)
        assert np.max(np.abs(gs[r, :gn[r]] - p[got]) / p[got]) < 1e-5
    assert near <= 2


# ------------------------------------------------------------------ 3. exact ties, also across a pass boundary
def test_exact_ties_across_a_pass_boundary(monkeypatch):
    """Items 100..139 (raw ids; internal 99..138, across the pass boundary at 128 below) get identical interaction
    columns, hence identical item-tower outputs and identical scores for every user.  The column is copied from the
    item that most users rank highest, so that the group lands in many top-k lists.  Tied items come out by id
    descending, and the answer equals the rank path, also with a pass boundary inside the group."""
    group = np.arange(100, 140)
    base = _data(6040, 3706, 400_000, seed=7)
    m0, _ = _model(base)
    top = m0.topk_batch(np.arange(m0.n_users, dtype=np.int32), 100, novelty=False)[0]
    cnt = np.bincount(top.ravel(), minlength=m0.n_items)
    cnt[[base.item_to_iid(x) for x in group]] = 0
    src_raw = base.iid_to_item(int(np.argmax(cnt)))

    def rows(u, i, v):                                     # the group's columns := the source item's column
        keep = ~np.isin(i, group)
        src = i == src_raw
        return (np.concatenate([u[keep], np.tile(u[src], len(group))]),
                np.concatenate([i[keep], np.repeat(group, src.sum())]),
                np.concatenate([v[keep], np.tile(v[src], len(group))]))
    ds = _data(6040, 3706, 400_000, seed=7, rows=rows)
    m, _ = _model(ds)
    g = np.array([ds.item_to_iid(x) for x in group])
    assert (np.sort(g) == g).all() and g.min() < 128 <= g.max()
    tied = np.append(g, ds.item_to_iid(src_raw))           # the source item scores the same as the group
    uids = np.arange(m.n_users, dtype=np.int32)
    ref = _rank_all(m, uids, True)
    for env in ({}, {'DRB_TOPK_CAP': '8192', 'DRB_TOPK_NS': str(m.n_items - 130)}):   # second: pass boundary at 128
        for key, val in env.items():
            monkeypatch.setenv(key, val)
        for k in (100, 2048):
            gi, gs, gn = _topk_raw(m, uids, k, True)
            _assert_same((gi, gs, gn), ref, k)
            seen_group = 0
            for r in range(m.n_users):
                row = gi[r, :gn[r]]
                t = row[np.isin(row, tied)]
                assert list(t) == sorted(t, reverse=True)
                if len(t) > 1:
                    assert len(set(gs[r, np.isin(row, tied)].tolist())) == 1      # one score for the whole group
                    seen_group += 1
            assert seen_group > 0


# ------------------------------------------------------------------ 4. the 1e-6 floor
def test_score_floor_keeps_the_lists_bounded(monkeypatch, c2):
    ds, _, w = c2
    w = {'user_nn': w['user_nn'], 'item_nn': [(k, b.copy()) for k, b in w['item_nn']]}
    w['item_nn'][-1] = (w['item_nn'][-1][0], np.full_like(w['item_nn'][-1][1], -1e3))   # item tower output: all zero
    m, _ = _model(ds, w=w)
    monkeypatch.setenv('DRB_TOPK_CAP', '1024')
    assert m.n_items > 1024
    uids = np.arange(0, m.n_users, 7, dtype=np.int32)
    (gi, gs, gn), prof = _profile(m, lambda: _topk_raw(m, uids, 100, True))
    assert 'k_dmf_topk_filter' in prof and 'k_dmf_fallback_scores' not in prof, prof
    for r, uid in enumerate(uids):
        alive = np.setdiff1d(np.arange(m.n_items), ds.user_items(int(uid)))
        assert gn[r] == 100 and gi[r].tolist() == alive[::-1][:100].tolist()
        assert (gs[r] == np.float32(1e-6)).all()
    _assert_same((gi, gs, gn), _rank_all(m, uids, True), 100)


# ------------------------------------------------------------------ 5. few eligible items
def test_user_with_few_unseen_items():
    def rows(u, i, v):
        extra = np.arange(41, 3707)                        # user 1 has seen every item but the first 40
        keep = u != 1
        return (np.concatenate([u[keep], np.full(len(extra), 1)]), np.concatenate([i[keep], extra]),
                np.concatenate([v[keep], np.full(len(extra), 3)]))
    ds = _data(600, 3706, 50000, seed=8, rows=rows)
    m, _ = _model(ds)
    uid = ds.user_to_uid(1)
    assert len(ds.user_items(uid)) == m.n_items - 40
    ref_on, ref_off = _rank_all(m, [uid], True), _rank_all(m, [uid], False)
    gi, gs, gn = _topk_raw(m, [uid], 100, True)
    assert gn[0] == 40
    _assert_same((gi, gs, gn), ref_on, 100)
    gi, gs, gn = _topk_raw(m, [uid], 100, False)
    assert gn[0] == 100
    _assert_same((gi, gs, gn), ref_off, 100)


# ------------------------------------------------------------------ 6. list overflow
def test_overflow_fallback_and_rerun(monkeypatch, wide):
    """A tiny list capacity and a first range of 128 items: tau is the 100th best of 128, so most of the catalog passes
    and most users overflow.  32 per block are re-done on the device, the rest come back as -1 and topk_batch re-runs
    them through the rank path.  The answer stays bitwise equal."""
    ds, m, _ = wide
    uids = np.arange(m.n_users, dtype=np.int32)
    ref = _rank_all(m, uids, True)
    monkeypatch.setenv('DRB_TOPK_CAP', '256')
    monkeypatch.setenv('DRB_TOPK_NS', '128')
    monkeypatch.setenv('DRB_TOPK_GROWTH', '1000')
    (gi, gs, gn), prof = _profile(m, lambda: _topk_raw(m, uids, 100, True))
    assert 'k_dmf_fallback_scores' in prof
    flagged = gn < 0
    assert flagged.sum() > m.n_users // 2
    ok = ~flagged
    _assert_same((gi[ok], gs[ok], gn[ok]), (ref[0][ok], ref[1][ok], ref[2][ok]), 100)
    ti, ts, tn = m.topk_batch(uids, 100, True)
    _assert_same((ti, ts, tn), (ref[0], m._rescale_value(ref[1]), ref[2]), 100)


# ------------------------------------------------------------------ 7. widths
@pytest.mark.parametrize('uf,itf', [([32, 16], [32, 16]), ([64, 48], [64, 48]), ([128, 64, 32], [64, 32])])
def test_tower_widths(uf, itf):
    ds = _data(500, 5000, 40000, seed=9)
    m, _ = _model(ds, uf, itf)
    uids = np.arange(m.n_users, dtype=np.int32)
    for novelty in (True, False):
        ref = _rank_all(m, uids, novelty)
        for k in (37, 100):
            _assert_same(_topk_raw(m, uids, k, novelty), ref, k)


# ------------------------------------------------------------------ 8. the item-tower cache
def test_cache_follows_the_weights():
    ds = _data(500, 4000, 40000, seed=11)
    m, w = _model(ds)
    uids = np.arange(m.n_users, dtype=np.int32)
    before = m.topk_batch(uids, 50, True)
    for s in range(1, 6):
        m._step = s
        m._train_step(64, 1e-4, want_loss=(s == 5))
    after = m.topk_batch(uids, 50, True)
    assert not np.array_equal(before[0], after[0])
    _assert_same(_topk_raw(m, uids, 50, True), _rank_all(m, uids, True), 50)
    m._store_epoch_weights(5)
    k, b = m.tower_weights('item_nn')[0]
    k.mul_(1.5)                                            # weight injection from Python
    _assert_same(_topk_raw(m, uids, 50, True), _rank_all(m, uids, True), 50)
    m._step = 6
    m._revert_weights(5)
    _assert_same(_topk_raw(m, uids, 50, True), _rank_all(m, uids, True), 50)
    np.testing.assert_array_equal(m.topk_batch(uids, 50, True)[0], after[0])


# ------------------------------------------------------------------ 9. public surface
def test_recommend_and_recommend_batch_dmf(c2, tmp_path):
    ds, m, _ = c2
    users = ds.raw_users[::301]
    # recommend() routes through topk_batch now and returns exactly what the rank route returned before
    for user in users[:6]:
        uid = ds.user_to_uid(user)
        old = [(r, ds.iid_to_item(i)) for r, i in m._rank(uid, range(m.n_items), 50, True)]
        new = m.recommend(user, n=50)
        assert new == old and [type(x[0]) for x in new] == [type(x[0]) for x in old]
    thr = float(m.recommend(users[0], n=20)[10][0])        # cuts the first user's list at 11 entries
    for t in (None, thr):
        items, scores, counts = m.recommend_batch(users, n=20, interaction_threshold=t)
        for r, user in enumerate(users):
            want = m.recommend(user, n=20, interaction_threshold=t)
            assert counts[r] == len(want)
            assert items[r, :counts[r]].tolist() == [it for _, it in want]
            assert scores[r, :counts[r]].tolist() == [s for s, _ in want]
            assert (items[r, counts[r]:] == -1).all()
        if t is not None:
            assert counts[0] >= 11 and (counts < 20).any()
    with pytest.raises(AssertionError, match='was not found'):
        m.recommend_batch([users[0], -12345], n=5)
    with pytest.raises(ValueError):
        m.recommend_batch(users, n=2049)
    p = str(tmp_path / 'dmf.joblib')
    m.save(p)
    m2 = drb.DMF.load(p)
    for a, b in zip(m.topk_batch(np.arange(200, dtype=np.int32), 30), m2.topk_batch(np.arange(200, dtype=np.int32), 30)):
        np.testing.assert_array_equal(a, b)


def test_recommend_batch_cdae_tensor_core_path():
    u, i, v = drb.synthetic_interactions(300, 9000, 40000, seed=6)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    m = drb.CDAE(hidden_factors=48, seed=10, verbose=False)
    m.fit(ds, epochs=0, batch_size=256)
    users = ds.raw_users[:200]                             # one block of >= 128 users: the tensor-core path
    items, scores, counts = m.recommend_batch(users, n=40)
    near = 0
    for r, user in enumerate(users[::13]):
        r *= 13
        want = m.recommend(user, n=40)
        assert counts[r] == len(want)
        got = items[r, :counts[r]].tolist()
        assert np.max(np.abs(scores[r, :counts[r]] - [s for s, _ in want]) / [s for s, _ in want]) < 1e-5
        if got != [it for _, it in want]:
            near += 1
    assert near <= 2


# ------------------------------------------------------------------ 10. errors
def test_errors(c2):
    ds, m, _ = c2
    uids = np.arange(10, dtype=np.int32)
    for k in (0, 2049):
        with pytest.raises(RuntimeError, match=r'k must be in \[1, 2048\]'):
            m.topk_batch(uids, k)
    with pytest.raises(RuntimeError, match='scratch'):
        _topk_raw(m, uids, 100, True, scratch_bytes=256)
