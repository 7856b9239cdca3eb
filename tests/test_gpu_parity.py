"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C-ABI / public API,
against the CPU oracle on identical seeded inputs, injected initial weights and sampler streams.

Tolerances are the ones BASELINE.json's north_star states: forward scores 1e-5 relative, loss after 100 steps
1e-3 relative, sampled pairs / index lists bit-exact (except documented near-ties)."""
import random

import numpy as np
import pytest

import drecpy_b200 as drb
from oracle import philox as ophilox
from oracle.cdae import CDAEOracle, corruption_keep_mt
from oracle.dmf import DMFOracle
from oracle.ranking import ranking_evaluation_oracle
from oracle.sampler import PointSamplerOracle

pytestmark = pytest.mark.gpu


def _dataset(U, I, nnz, seed=10):
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=seed)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    return ds


def _cdae_weights(U, I, K, seed=1, scale=1.0):
    rng = np.random.default_rng(seed)

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo)) * scale
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    return {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K),
            'b': glorot((K,), K, K), 'b_': glorot((I,), I, I)}


def _make_cdae(ds, K, B, w, **kw):
    m = drb.CDAE(hidden_factors=K, corruption_level=kw.pop('q', 0.2), loss=kw.pop('loss', 'bce'), seed=10,
                 verbose=False, **kw)
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=1e-3, init_weights=w)
    return m


def _oracle_cdae(ds, w, **kw):
    return CDAEOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), interaction_threshold=1e-3,
                      learning_rate=1e-3, **kw)


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


@pytest.mark.parametrize('K', [50, 64, 130, 200])
def test_cdae_forward_scores(K):
    U, I = 300, 1682 if K == 50 else 777
    ds = _dataset(U, I, 12000)
    w = _cdae_weights(U, I, K, scale=3.0)
    m = _make_cdae(ds, K, 32, w)
    o = _oracle_cdae(ds, w)
    uids = np.array([0, 5, 17, 299, 123, 5])
    h = m.hidden(uids)
    assert rel_err(h, o.hidden(uids)) < 1e-5
    for uid in (0, 17, 299):
        p, po = m._predict(uid), o.predict(uid)
        assert p.shape == (I,)
        assert np.max(np.abs(p - po) / np.abs(po)) < 1e-5          # forward scores within 1e-5 relative
    assert abs(m.predict(ds.uid_to_user(17), ds.iid_to_item(3)) - o.predict(17)[3]) <= 1e-5 * o.predict(17)[3]


def _run_cdae_steps(ds, K, B, steps, oracle_kw, model_kw, mask='mt19937', reg=1e-3):
    U, I = ds.count_unique('uid'), ds.count_unique('iid')
    w = _cdae_weights(U, I, K)
    m = _make_cdae(ds, K, B, w, rng_mode=mask, **model_kw)
    o = _oracle_cdae(ds, w, **oracle_kw)
    so = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10)
    pr = random.Random(10)
    losses, losses_o = [], []
    pos = ds.csr(1e-3)
    for s in range(1, steps + 1):
        m._step = s
        losses.append(m._train_step(B, reg, want_loss=True))
        triples = so.sample(B)
        uids = np.array([t[0] for t in triples])
        if mask == 'mt19937':
            keep = np.stack([corruption_keep_mt(pr, I, o.q) for _ in uids])
        else:
            keep = np.ones((B, I), bool)
            for b, u in enumerate(uids):
                items = pos[1][pos[0][u]:pos[0][u + 1]]
                keep[b, items] = ophilox.keep_mask(items, b, s, 10, o.q)
        losses_o.append(float(o.step(uids, keep, reg)))
    return m, o, np.array(losses), np.array(losses_o)


def test_cdae_100_steps_config1():
    """C1: 943 x 1682, 100k interactions, K=50, q=0.2, bce, B=64, neg_ratio=5, seed=10, reference-faithful modes."""
    ds = _dataset(943, 1682, 100000)
    m, o, l, lo = _run_cdae_steps(ds, 50, 64, 100, {}, {})
    assert np.all(np.isfinite(l))
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3, (l[-5:], lo[-5:])       # every step, not only step 100
    assert abs(l[-1] - lo[-1]) / abs(lo[-1]) < 1e-3
    for name in ('W', 'V', 'b', 'b_'):
        got = getattr(m, name).cpu().numpy()
        assert rel_err(got, getattr(o, name)) < 2e-3, name
    assert rel_err(m.W_.cpu().numpy(), o.W_) < 2e-3


@pytest.mark.parametrize('case', ['per_user', 'mse', 'mse_per_user', 'philox', 'per_step_adam', 'q0'])
def test_cdae_step_modes(case):
    ds = _dataset(211, 389, 9000, seed=4)
    okw, mkw, mask = {}, {}, 'mt19937'
    if case == 'per_user': okw, mkw = {'label_mode': 'per_user'}, {'label_mode': 'per_user'}
    if case == 'mse': okw, mkw = {'loss': 'mse'}, {'loss': 'mse'}
    if case == 'mse_per_user':
        okw, mkw = {'loss': 'mse', 'label_mode': 'per_user'}, {'loss': 'mse', 'label_mode': 'per_user'}
    if case == 'philox': mask = 'philox'
    if case == 'per_step_adam': okw, mkw = {'adam_t': 'per_step'}, {'adam_t': 'per_step'}
    if case == 'q0': okw, mkw = {'corruption_level': 0.0}, {'q': 0.0}
    m, o, l, lo = _run_cdae_steps(ds, 36, 48, 25, okw, mkw, mask=mask)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3, (case, l[-3:], lo[-3:])
    assert rel_err(m.W.cpu().numpy(), o.W) < 2e-3
    assert rel_err(m.V.cpu().numpy(), o.V) < 2e-3


def test_cdae_empty_rows_duplicate_rows_and_batch_of_one():
    """interaction_threshold=4 leaves many users without a single positive (empty CSR rows); the raw data also holds
    duplicated (user, item) rows, which the reference sums before thresholding (mem_dataset.py:495, cdae.py:61)."""
    import torch
    rng = np.random.default_rng(3)
    u, i, v = drb.synthetic_interactions(90, 140, 700, seed=11)
    dup = rng.choice(len(u), 60, replace=False)
    u, i, v = np.concatenate([u, u[dup]]), np.concatenate([i, i[dup]]), np.concatenate([v, rng.integers(1, 3, 60)])
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    U, I, K = ds.count_unique('uid'), ds.count_unique('iid'), 12
    w = _cdae_weights(U, I, K)
    m = drb.CDAE(hidden_factors=K, corruption_level=0.0, seed=10, verbose=False, interaction_threshold=4,
                 rng_mode='philox')
    m.fit(ds, epochs=0, batch_size=8, init_weights=w)
    o = CDAEOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), interaction_threshold=4, corruption_level=0.0,
                   learning_rate=1e-3)
    deg = np.diff(ds.csr(4)[0])
    assert (deg == 0).any() and (deg > 0).any()
    empty, full = int(np.flatnonzero(deg == 0)[0]), int(deg.argmax())
    for uids in (np.array([empty], np.int32), np.array([full, empty, empty, 3, full], np.int32)):
        off = np.concatenate([[0], np.cumsum(deg[uids])]).astype(np.int32)
        loss = torch.zeros(2, device='cuda')
        m.step_device(torch.as_tensor(uids, device='cuda'), torch.as_tensor(off, device='cuda'), None, 1e-3, loss)
        lo = o.step(uids, np.ones((len(uids), I), bool), 1e-3)
        assert abs(loss[0].item() - lo) / abs(lo) < 1e-5
    assert rel_err(m.V.cpu().numpy(), o.V) < 1e-4 and rel_err(m.W.cpu().numpy(), o.W) < 1e-4
    assert np.max(np.abs(m._predict(empty) - o.predict(empty)) / o.predict(empty)) < 1e-5


def test_cdae_duplicate_users_and_ragged_rows():
    """batch with repeated users, a user with a single interaction and the largest-degree user."""
    ds = _dataset(150, 260, 5000, seed=8)
    U, I, K = 150, 260, 20
    w = _cdae_weights(U, I, K)
    m = _make_cdae(ds, K, 16, w, rng_mode='philox', q=0.0)
    o = _oracle_cdae(ds, w, corruption_level=0.0)
    deg = np.diff(ds.csr(1e-3)[0])
    import torch
    uids = np.array([3, 3, 3, int(deg.argmax()), int(deg.argmin()), 9, 9, 0, 149, 149, 77, 3], np.int32)
    off = np.concatenate([[0], np.cumsum(deg[uids])]).astype(np.int32)
    loss = torch.zeros(2, device='cuda')
    m.step_device(torch.as_tensor(uids, device='cuda'), torch.as_tensor(off, device='cuda'), None, 1e-3, loss)
    lo = o.step(uids, np.ones((len(uids), I), bool), 1e-3)
    assert abs(loss[0].item() - lo) / abs(lo) < 1e-5
    assert rel_err(m.V.cpu().numpy(), o.V) < 1e-4
    assert rel_err(m.W.cpu().numpy(), o.W) < 1e-4


def test_cdae_batch_larger_than_one_scan_tile():
    """B = 4500 sampled users: the piece-map scan (k_chunk_scan) walks more than one 4096-row tile and carries the
    running total across; loss and weights against the oracle."""
    ds = _dataset(211, 389, 9000, seed=4)
    m, o, l, lo = _run_cdae_steps(ds, 16, 4500, 2, {}, {}, mask='philox')
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-4, (l, lo)
    assert rel_err(m.W.cpu().numpy(), o.W) < 5e-4 and rel_err(m.V.cpu().numpy(), o.V) < 5e-4


@pytest.mark.parametrize('mask', ['mt19937', 'philox'])
def test_cdae_heavy_rows_span_several_pieces(mask):
    """Users with 300..1400 interactions: the balanced gather / scatter of the training step cut their CSR rows into
    256-entry pieces (sparse.cu: k_gather_chunks / k_scatter_chunks); the corruption mask bytes of a piece start at
    keep_off[b] + 256 * piece.  Loss and weights against the oracle, every step."""
    rng = np.random.default_rng(5)
    U, I = 40, 1500
    deg = rng.integers(300, 1400, U)
    deg[:3] = [1, 256, 257]                               # piece boundaries
    u = np.repeat(np.arange(U), deg)
    i = np.concatenate([rng.choice(I, d, replace=False) for d in deg])
    perm = rng.permutation(len(u))
    ds = drb.InteractionData(u[perm] + 1, i[perm] + 1, rng.integers(1, 6, len(u)))
    ds.assign_internal_ids()
    m, o, l, lo = _run_cdae_steps(ds, 24, 32, 6, {}, {}, mask=mask)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-4, (l, lo)
    for name in ('W', 'V', 'b', 'b_'):
        assert rel_err(getattr(m, name).cpu().numpy(), getattr(o, name)) < 5e-4, name
    assert rel_err(m.W_.cpu().numpy(), o.W_) < 5e-4


def _dmf_weights(U, I, uf, itf, seed=2):
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


@pytest.mark.parametrize('uf,itf,l2n,nce', [([64, 32], [64, 32], True, True), ([50], [24, 50], True, False),
                                            ([40, 20, 12], [64, 12], False, True)])
def test_dmf_steps_and_scores(uf, itf, l2n, nce):
    U, I, B = 400, 600, 64
    ds = _dataset(U, I, 20000, seed=5)
    w = _dmf_weights(U, I, uf, itf)
    m = drb.DMF(user_factors=uf, item_factors=itf, use_nce=nce, l2_norm_vectors=l2n, seed=10, verbose=False)
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=1e-4, init_weights=w)
    o = DMFOracle(w['user_nn'], w['item_nn'], ds.csr(), ds.csc(), m.min_interaction, m.max_interaction,
                  use_nce=nce, l2_norm_vectors=l2n, learning_rate=1e-3)
    uids, iids = np.array([0, 3, 399, 17, 17]), np.array([5, 599, 0, 44, 45])
    p, po = m.forward_pairs(uids, iids), o.forward(uids, iids)[0]
    assert np.max(np.abs(p - po) / np.abs(po)) < 1e-5
    assert abs(m._predict(3, 599) - o.predict(3, 599)) < 1e-5 * abs(o.predict(3, 599))
    so = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10)
    l, lo = [], []
    for s in range(1, 41):
        m._step = s
        l.append(m._train_step(B, 1e-4, want_loss=True))
        t = so.sample(B)
        labels = [o.standardize(x[2]) if nce else x[2] for x in t]
        lo.append(float(o.step([x[0] for x in t], [x[1] for x in t], labels, 1e-4)))
    l, lo = np.array(l), np.array(lo)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3, (l[-3:], lo[-3:])
    for (k, b), (ko, bo) in zip(m.tower_weights('user_nn') + m.tower_weights('item_nn'),
                                o.user_layers + o.item_layers):
        assert rel_err(k.cpu().numpy(), ko) < 2e-3
        assert rel_err(b.cpu().numpy(), bo) < 2e-3


def test_dmf_graph_replay_equals_direct_launches(monkeypatch):
    """drb_dmf_step replays an instantiated CUDA graph (the step is launch bound); DRB_GRAPH=0 launches every kernel
    directly.  Same kernels in the same order: losses and weights agree to the last bits (the scatter kernels add
    with atomics, so not bit for bit) and the launch counts match."""
    U, I, B = 300, 500, 64
    ds = _dataset(U, I, 15000, seed=8)
    w = _dmf_weights(U, I, [64, 32], [64, 32])
    runs = []
    for graph in ('1', '0'):
        monkeypatch.setenv('DRB_GRAPH', graph)
        m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
        m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=1e-4, init_weights=w)
        n0 = m.launch_count()
        losses = []
        for s in range(1, 13):
            m._step = s
            losses.append(m._train_step(B if s % 5 else B // 2, 1e-4, want_loss=True))   # a second batch size: second graph
        runs.append((losses, m.launch_count() - n0, [k.cpu().numpy() for k, _ in m.tower_weights('user_nn')]))
    assert np.allclose(runs[0][0], runs[1][0], rtol=2e-6, atol=0)
    # graph mode adds one k_set_scalars launch per step
    assert runs[0][1] == runs[1][1] + 12
    for a, b in zip(runs[0][2], runs[1][2]):
        assert rel_err(a, b) < 1e-5


@pytest.mark.parametrize('mask', ['mt19937', 'philox'])
def test_cdae_graph_replay_equals_direct_launches(monkeypatch, mask):
    """The ml-100k-sized step is launch bound: from the second step on drb_cdae_step replays an instantiated CUDA graph
    (per-step scalars -- five Adam step sizes, philox step -- read from device memory).  DRB_GRAPH=0 launches every
    kernel.  Same kernels, same order: the losses agree to the last bits and so do the weights."""
    ds = _dataset(300, 500, 15000, seed=8)
    w = _cdae_weights(300, 500, 24)
    runs = []
    for graph in ('1', '0'):
        monkeypatch.setenv('DRB_GRAPH', graph)
        m = _make_cdae(ds, 24, 48, w, rng_mode=mask)
        n0 = m.launch_count()
        losses = []
        for s in range(1, 13):
            m._step = s
            losses.append(m._train_step(48 if s % 5 else 32, 1e-3, want_loss=True, prefetch=True))
        runs.append((losses, m.launch_count() - n0, m._params.cpu().numpy()))
    assert np.allclose(runs[0][0], runs[1][0], rtol=2e-6, atol=0), (runs[0][0], runs[1][0])
    assert runs[0][1] > runs[1][1]                 # graph mode: one extra k_set_scalars per replayed step
    assert rel_err(runs[0][2], runs[1][2]) < 1e-5
    # and the graph path still matches the oracle over many steps
    monkeypatch.setenv('DRB_GRAPH', '1')
    m, o, l, lo = _run_cdae_steps(ds, 24, 48, 30, {}, {}, mask=mask)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3


@pytest.mark.parametrize('model', ['cdae', 'dmf'])
def test_graph_capture_cap_and_slot_replacement(monkeypatch, model):
    """How a model keeps its step graphs.  Cap: a new reg_rate every step is a new argument set every step, so every
    step is a capture; after 32 captures the model gives up on graphs and launches directly.  Replacement: ten batch
    sizes, cycled twice, through the eight graph slots.  Either way graph mode computes what direct launches compute
    and adds one k_set_scalars launch per replayed step (CDAE's first step runs directly: dV is not yet known clean)."""
    U, I = 300, 500
    ds = _dataset(U, I, 15000, seed=8)
    if model == 'cdae':
        B, reg, w = 48, 1e-3, _cdae_weights(U, I, 24)
    else:
        B, reg, w = 64, 1e-4, _dmf_weights(U, I, [64, 32], [64, 32])

    def make():
        if model == 'cdae':
            return _make_cdae(ds, 24, B, w)
        m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
        m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=reg, init_weights=w)
        return m
    first_direct = 1 if model == 'cdae' else 0
    cap = [(B, reg * (1 + s / 64)) for s in range(40)]
    cycle = [(B - 4 * j, reg) for j in range(10)] * 2
    for steps, replayed in ((cap, 32), (cycle, len(cycle) - first_direct)):
        runs = []
        for graph in ('1', '0'):
            monkeypatch.setenv('DRB_GRAPH', graph)
            m = make()
            n0 = m.launch_count()
            losses = []
            for s, (b, r) in enumerate(steps, 1):
                m._step = s
                losses.append(m._train_step(b, r, want_loss=True))
            runs.append((losses, m.launch_count() - n0, m._params.cpu().numpy()))
        assert np.allclose(runs[0][0], runs[1][0], rtol=2e-6, atol=0), (runs[0][0], runs[1][0])
        assert runs[0][1] == runs[1][1] + replayed
        assert rel_err(runs[0][2], runs[1][2]) < 1e-5


@pytest.mark.parametrize('loss,K', [('bce', 36), ('mse', 200)])
def test_cdae_sampled_output_steps_vs_oracle(loss, K):
    """The sampled-output extension (BASELINE configs[4]'s mode): positives + 2 groups x 20 drawn items per sampled
    user instead of the whole catalog, against oracle.cdae.CDAESampledOracle (same philox draws): every loss within
    1e-4, weights within 5e-4 of their scale."""
    from oracle.cdae import CDAESampledOracle
    ds = _dataset(211, 389, 9000, seed=4)
    U, I, B = 211, 389, 48
    w = _cdae_weights(U, I, K)
    m = _make_cdae(ds, K, B, w, rng_mode='philox', output='sampled', neg_per_group=20, neg_groups=2, loss=loss)
    o = CDAESampledOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), interaction_threshold=1e-3,
                          learning_rate=1e-3, loss=loss, n_groups=2, neg_per_group=20, seed=10)
    so = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10)
    pos = ds.csr(1e-3)
    l, lo = [], []
    for s in range(1, 16):
        m._step = s
        l.append(m._train_step(B, 1e-3, want_loss=True))
        uids = np.array([t[0] for t in so.sample(B)])
        keep = np.ones((B, I), bool)
        for b, u in enumerate(uids):
            items = pos[1][pos[0][u]:pos[0][u + 1]]
            keep[b, items] = ophilox.keep_mask(items, b, s, 10, o.q)
        lo.append(float(o.step_sampled(uids, keep, 1e-3, s)))
    l, lo = np.array(l), np.array(lo)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-4, (l, lo)
    for name in ('W', 'V', 'b', 'b_'):
        assert rel_err(getattr(m, name).cpu().numpy(), getattr(o, name)) < 5e-4, name
    assert rel_err(m.W_.cpu().numpy(), o.W_) < 5e-4
    # scoring of a sampled-output model still works (dense predict, candidate ranking)
    p = m._predict(7)
    assert p.shape == (I,) and np.all((p > 0) & (p < 1))
    assert len(m._rank(7, list(range(0, I, 5)), 20, True)) == 20


def test_rank_order_ties_and_novelty():
    """(score desc, iid desc) == heapq.nlargest on (score, iid) tuples (cdae.py:102-103), duplicates collapsed,
    training items dropped when novelty."""
    U, I, K = 120, 333, 16
    ds = _dataset(U, I, 4000, seed=6)
    w = _cdae_weights(U, I, K)
    w['W_'][:, 100:140] = w['W_'][:, 100:101]          # forced exact score ties among items 100..139
    w['b_'][100:140] = w['b_'][100]
    m = _make_cdae(ds, K, 16, w)
    o = _oracle_cdae(ds, w)
    rng = np.random.default_rng(0)
    for uid in (0, 7, 119):
        cand = rng.choice(I, 101, replace=False).tolist() + list(range(100, 140)) + [5, 5, 6]
        for novelty in (True, False):
            got = m._rank(uid, cand, len(cand), novelty)
            want = o.rank(uid, cand, len(cand), novelty)
            assert [i for _, i in got] == [i for _, i in want]
            assert np.allclose([s for s, _ in got], [s for s, _ in want], rtol=1e-5)
        top = m._recommend(uid, 50, True, None)
        want = o.rank(uid, range(I), 50, True)
        assert [i for _, i in top] == [i for _, i in want]
    oi, os_, on = m.topk_batch(np.arange(U, dtype=np.int32), 100, novelty=True)
    for uid in range(0, U, 13):
        want = o.rank(uid, range(I), 100, True)
        assert oi[uid, :on[uid]].tolist() == [i for _, i in want]
    # whole-catalog ranking longer than the in-CTA sorter (recommend(n=None)): same order, device-side sort
    I_big = 5000
    ds2 = _dataset(60, I_big, 3000, seed=7)
    w2 = _cdae_weights(60, I_big, 8)
    w2['W_'][:, 10:30] = w2['W_'][:, 10:11]
    w2['b_'][10:30] = w2['b_'][10]
    m2 = _make_cdae(ds2, 8, 8, w2)
    o2 = _oracle_cdae(ds2, w2)
    got = m2.recommend(ds2.uid_to_user(5))
    want = o2.rank(5, range(I_big), I_big, True)
    got_i = [ds2.item_to_iid(it) for _, it in got]
    assert sorted(got_i) == sorted(i for _, i in want)
    po = o2.predict(5)
    so = po[got_i]                              # oracle scores in the GPU's order: non-increasing up to fp32 noise,
    assert np.all(so[:-1] >= so[1:] * (1 - 1e-6))
    forced = [i for i in got_i if 10 <= i < 30]  # ... and the forced exact ties by item id descending
    assert len(forced) >= 10 and forced == sorted(forced, reverse=True)
    # k larger than the number of eligible items
    got = m.rank(ds.uid_to_user(3), [ds.iid_to_item(x) for x in (1, 2, 3)], novelty=False)
    assert len(got) == 3


def test_ranking_evaluation_native_cdae_vs_oracle():
    U, I, K = 200, 300, 24
    u, i, v = drb.synthetic_interactions(U, I, 9000, seed=12)
    rng = np.random.default_rng(1)
    test_mask = np.zeros(len(u), bool)
    for usr in np.unique(u):                     # leave-1-out style split
        idx = np.flatnonzero(u == usr)
        if len(idx) > 3: test_mask[rng.choice(idx)] = True
    train = drb.InteractionData(u[~test_mask], i[~test_mask], v[~test_mask])
    test = drb.InteractionData(u[test_mask], i[test_mask], v[test_mask])
    train.assign_internal_ids()
    w = _cdae_weights(train.count_unique('uid'), train.count_unique('iid'), K, scale=4.0)
    m = drb.CDAE(hidden_factors=K, seed=10, verbose=False)
    m.fit(train, epochs=3, batch_size=32, init_weights=w)
    o = CDAEOracle(m.W.cpu().numpy(), m.W_.cpu().numpy(), m.V.cpu().numpy(), m.b.cpu().numpy(),
                   m.b_.cpu().numpy(), train.csr(), interaction_threshold=1e-3)

    def rank_fn(user, items, novelty):
        uid = train.user_to_uid(user)
        iids = [x for x in (train.item_to_iid(it) for it in items) if x is not None]
        return [train.iid_to_item(i) for _, i in o.rank(uid, iids, len(iids), novelty)]
    train_pos = {}
    for a, b, c in zip(train.user.tolist(), train.item.tolist(), train.interaction.tolist()):
        if c >= 1e-3: train_pos.setdefault(a, set()).add(b)
    kw = dict(k=[1, 5, 10], n_pos_interactions=1, n_neg_interactions=100, generate_negative_pairs=True, novelty=True,
              seed=10)
    rec, rec_o = [], []
    got = drb.ranking_evaluation(m, test, metrics=[drb.HitRatio(), drb.NDCG()], record=rec, verbose=False, **kw)
    want = ranking_evaluation_oracle(rank_fn, test.user.tolist(), test.item.tolist(), test.interaction.tolist(),
                                     train_pos, m.n_items, 1e-3, metrics=('HitRatio', 'NDCG'), record=rec_o, **kw)
    assert [r[1] for r in rec] == [r[1] for r in rec_o]           # candidate lists bit-exact
    mism = sum(r[2] != ro[2] for r, ro in zip(rec, rec_o))
    assert mism <= max(1, len(rec) // 100), mism                    # ranked lists: documented near-ties only
    if mism == 0:
        assert got == want
    else:
        assert all(abs(got[k_] - want[k_]) < 5e-3 for k_ in want)


def test_fit_public_api_callbacks_early_stopping_and_save_load(tmp_path):
    ds = _dataset(120, 200, 4000, seed=9)
    calls = []

    def cb(model):
        calls.append(model._step)
        return {'val_HitRatio@10': [0.1, 0.5, 0.3, 0.2][len(calls) - 1]}
    m = drb.CDAE(hidden_factors=12, seed=10, verbose=False)
    m.fit(ds, epochs=20, batch_size=16, epoch_callback_fn=cb, epoch_callback_freq=5,
          early_stopping_rule=drb.MaxValidationValueRule('val_HitRatio'), early_stopping_freq=5)
    assert calls == [5, 10, 15, 20]
    assert len(m._loss_tracker.epoch_losses) == 20 and m._loss_tracker.called_epochs == [5, 10, 15, 20]
    # best epoch = 10 -> weights reverted to the snapshot taken at epoch 10
    assert np.array_equal(m._params.cpu().numpy(), m.epoch_weights[10].cpu().numpy())
    p = m.predict(ds.uid_to_user(0), ds.iid_to_item(0))
    path = str(tmp_path / 'model.joblib')
    m.save(path)
    m2 = drb.CDAE.load(path)
    assert abs(m2.predict(ds.uid_to_user(0), ds.iid_to_item(0)) - p) < 1e-7
    with pytest.raises(AssertionError, match='User 999999 was not found.'):
        m.predict(999999, ds.iid_to_item(0))
    assert m.predict(999999, ds.iid_to_item(0), skip_errors=True) is None
    with pytest.raises(Exception, match='Loss function "hinge" is not supported'):
        drb.CDAE(loss='hinge')


def test_dmf_fit_rank_and_save_load(tmp_path):
    ds = _dataset(150, 220, 5000, seed=13)
    m = drb.DMF(user_factors=[32, 16], item_factors=[32, 16], seed=10, verbose=False)
    m.fit(ds, epochs=15, batch_size=64, learning_rate=1e-3, reg_rate=1e-4)
    user, items = ds.uid_to_user(4), [ds.iid_to_item(x) for x in (3, 50, 7, 120, 199)]
    ranked = m.rank(user, items, novelty=False)
    assert len(ranked) == 5 and all(ranked[j][0] >= ranked[j + 1][0] for j in range(4))
    preds = {it: m.predict(user, it) for it in items}
    for s, it in ranked:
        assert abs(s - preds[it]) <= 1e-5 * max(abs(preds[it]), 1e-6)     # rank() reports the rescaled prediction
    path = str(tmp_path / 'dmf.joblib')
    m.save(path)
    m2 = drb.DMF.load(path)
    assert abs(m2.predict(user, items[0]) - preds[items[0]]) < 1e-7
    res = drb.ranking_evaluation(m2, ds, k=5, n_pos_interactions=1, n_neg_interactions=20, generate_negative_pairs=True,
                                 novelty=False, metrics=[drb.HitRatio(), drb.NDCG()], verbose=False)
    assert set(res) == {'HitRatio@5', 'NDCG@5'} and 0 <= res['HitRatio@5'] <= 1
