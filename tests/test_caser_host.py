"""Caser host side (no GPU): the float64 oracle's hand-written backward pass against torch.autograd, the window /
negative sampler replay, and timestamps through InteractionData and leave_k_out."""
import numpy as np
import pandas as pd
import pytest
import torch

import drecpy_b200 as drb
from oracle import caser as oc


def _weights(rng, n_users, n_items, L, d, n_v, n_h):
    F = n_v * d + n_h * L
    return {'E': rng.normal(0, .3, (n_items, d)), 'P': rng.normal(0, .3, (n_users, d)), 'Fv': rng.normal(0, .5, (L, n_v)),
            'bv': rng.normal(0, .1, n_v), 'Fh': [rng.normal(0, .3, (h, d, n_h)) for h in range(1, L + 1)],
            'bh': [rng.normal(0, .1, n_h) for _ in range(L)], 'fc': rng.normal(0, .2, (F, d)), 'bfc': rng.normal(0, .1, d),
            'W2': rng.normal(0, .3, (n_items, 2 * d)), 'b2': rng.normal(0, .1, n_items)}


def _torch_loss(w, users, items, L, T, scale, reg):
    """Caser forward + loss written with torch ops (autograd gives the gradients)."""
    E, P = w['E'], w['P']
    inp, tgt = items[:, :L], items[:, L:]
    eh = E[torch.as_tensor(inp)]
    ov = torch.einsum('lc,bld->bcd', w['Fv'], eh) + w['bv'][None, :, None]
    oh = []
    for h in range(1, L + 1):
        conv = torch.stack([torch.einsum('bqd,qdf->bf', eh[:, i:i + h], w['Fh'][h - 1]) for i in range(L - h + 1)], 1)
        oh.append(torch.relu(conv + w['bh'][h - 1]).max(dim=1).values)
    c = torch.cat([ov.reshape(len(users), -1)] + oh, 1) * torch.as_tensor(scale)
    z = torch.relu(c @ w['fc'] + w['bfc'])
    x = torch.cat([z, P[torch.as_tensor(users, dtype=torch.long)]], 1)
    t_ = torch.as_tensor(tgt, dtype=torch.long)
    y = torch.einsum('bk,bjk->bj', x, w['W2'][t_]) + w['b2'][t_]
    t = torch.zeros_like(y)
    t[:, :T] = 1
    p = torch.sigmoid(y)
    pc = p.clamp(oc.KERAS_EPS, 1 - oc.KERAS_EPS)
    loss = -(t * torch.log(pc + oc.KERAS_EPS) + (1 - t) * torch.log(1 - pc + oc.KERAS_EPS)).mean()
    for k in oc.L2_TENSORS:
        for v in (w[k] if isinstance(w[k], list) else [w[k]]):
            loss = loss + reg * (v ** 2).sum()
    return loss


@pytest.mark.parametrize('L,T,d,n_v,n_h,rate', [(5, 3, 50, 4, 16, 0.5), (3, 1, 20, 2, 3, 0.0)])
def test_oracle_backward_matches_autograd(L, T, d, n_v, n_h, rate):
    rng = np.random.default_rng(L * 7 + d)
    U, I, B, neg = 9, 40, 6, 2
    w = _weights(rng, U, I, L, d, n_v, n_h)
    users = rng.integers(0, U, B)
    items = rng.integers(0, I, (B, L + T * (1 + neg)))
    scale = oc.dropout_scale(n_v * d + n_h * L, B, 77, 3, rate)
    o = oc.CaserOracle(w)
    loss, g, _ = o.loss_and_grads(users, items, L, T, scale, 0.01)
    tw = {k: ([torch.tensor(x, requires_grad=True) for x in v] if isinstance(v, list) else torch.tensor(v, requires_grad=True))
          for k, v in w.items()}
    tl = _torch_loss(tw, users, items, L, T, scale, 0.01)
    tl.backward()
    assert abs(tl.item() - loss) < 1e-12
    for k, v in tw.items():
        for j, t_ in enumerate(v if isinstance(v, list) else [v]):
            want = t_.grad.numpy() - (2 * 0.01 * t_.detach().numpy() if k in oc.L2_TENSORS else 0)
            got = g[k][j] if isinstance(v, list) else g[k]
            np.testing.assert_allclose(got, want, rtol=1e-9, atol=1e-12, err_msg=k)


def _seq_data(seed=3):
    rng = np.random.default_rng(seed)
    n = 400
    u = rng.integers(0, 20, n)
    i = rng.integers(0, 60, n)
    ts = rng.integers(0, 1000, n)
    return u, i, ts


def test_sampler_replay():
    u, i, ts = _seq_data()
    ds = drb.InteractionData(u, i, np.ones(len(u)), timestamp=ts)
    ds.assign_internal_ids()
    U, I = ds.count_unique('uid'), ds.count_unique('iid')
    L, T, neg = 5, 3, 4
    indptr, seq = oc.sequences(ds.uid, ds.iid, ds.interaction, U, None, ds.timestamp)
    win = oc.window_offsets(indptr, L, T)
    seen = ds.csr()[:2]
    a = oc.sample_batch(indptr, seq, win, seen, I, L, T, neg, 64, 123, 7)
    b = oc.sample_batch(indptr, seq, win, seen, I, L, T, neg, 64, 123, 7)
    c = oc.sample_batch(indptr, seq, win, seen, I, L, T, neg, 64, 124, 7)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert not np.array_equal(a[1], c[1])
    users, items = a
    for b_, uu in enumerate(users):
        s = seq[indptr[uu]:indptr[uu + 1]].tolist()
        assert len(s) >= L + T
        row = items[b_, :L + T].tolist()
        assert any(s[j:j + L + T] == row for j in range(len(s) - L - T + 1))          # a full window
        stored = set(seen[1][seen[0][uu]:seen[0][uu + 1]].tolist())
        if len(stored) < I:
            assert not (set(items[b_, L + T:].tolist()) & stored)


def test_sequences_follow_timestamps_then_rows():
    u = np.array([0, 0, 0, 1, 0])
    i = np.array([1, 2, 3, 4, 5])
    ts = np.array([5, 1, 5, 0, 0])
    indptr, seq = oc.sequences(u, i, np.ones(5), 2, None, ts)
    assert seq[indptr[0]:indptr[1]].tolist() == [5, 2, 1, 3]
    indptr, seq = oc.sequences(u, i, np.ones(5), 2, None, None)
    assert seq[indptr[0]:indptr[1]].tolist() == [1, 2, 3, 5]


def test_timestamps_round_trip():
    u, i, ts = _seq_data(5)
    v = np.ones(len(u))
    df = pd.DataFrame({'user': u, 'item': i, 'interaction': v, 'ts': ts})
    ds = drb.InteractionData.read_df(df, timestamp_label='ts')
    assert np.array_equal(ds.timestamp, ts)
    assert drb.InteractionData.read_df(df).timestamp is None
    class Frame:
        _df = df.rename(columns={'ts': 'timestamp'})
    assert np.array_equal(drb.InteractionData.from_dataset(Frame()).timestamp, ts)
    for last in (False, True):
        tr, te = drb.leave_k_out(ds, k=2, last_timestamps=last, seed=3)
        plain_tr, plain_te = drb.leave_k_out(drb.InteractionData(u, i, v), k=2, seed=3) if not last else (tr, te)
        for part in (tr, te):
            key = dict(zip(zip(u.tolist(), i.tolist(), ts.tolist()), range(len(u))))
            assert all((a, b, c) in key for a, b, c in zip(part.user.tolist(), part.item.tolist(), part.timestamp.tolist()))
        assert np.array_equal(tr.user, plain_tr.user) and np.array_equal(te.item, plain_te.item)
        assert plain_tr.timestamp is None or last
