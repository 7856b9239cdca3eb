"""Host-side interaction table: the members of DRecPy's InteractionDataset that the hot path touches.

Mirrors (reference, DRecPy/Dataset/):
  mem_dataset.py:309-330   assign_internal_ids  (ids = order of first appearance)
  mem_dataset.py:480-498   _build_interaction_matrix  (CSR, duplicates summed, column-sorted) -- here a one-pass
                           sort instead of the reference's O(users * nnz) Python loop
  mem_dataset.py:165-218   select_user_interaction_vec / select_item_interaction_vec
  dataset_abc.py           user_to_uid / uid_to_user / item_to_iid / iid_to_item / count_unique / min / max
Storage, querying and file IO of the reference dataset classes are out of scope (SURVEY.md section 8); a
reference InteractionDataset object can be passed to fit() directly and is converted with `from_dataset`.
"""
import numpy as np
import pandas as pd


def _build_csr(rows, cols, vals, n_rows, n_cols):
    rows = np.asarray(rows, np.int64)
    cols = np.asarray(cols, np.int64)
    vals = np.asarray(vals, np.float64)
    if len(rows) == 0:
        return np.zeros(n_rows + 1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.float64)
    key = rows * n_cols + cols
    order = _argsort_stable(key)
    key_s = key[order]
    starts = np.flatnonzero(np.concatenate(([True], key_s[1:] != key_s[:-1])))
    data = np.add.reduceat(vals[order], starts)          # duplicates summed (scipy csr_matrix semantics)
    ukey = key_s[starts]
    r = ukey // n_cols
    indptr = np.zeros(n_rows + 1, np.int64)
    np.cumsum(np.bincount(r, minlength=n_rows), out=indptr[1:])
    return indptr, (ukey % n_cols).astype(np.int32), data


def _argsort_stable(keys):
    """np.argsort(kind='stable') for large integer arrays through torch's multi-threaded CPU sort (same permutation:
    both are stable); ~6x faster at 2e7 keys, which is the whole cost of building the CSR views of an ml-20m table."""
    keys = np.ascontiguousarray(keys)
    if len(keys) < 1_000_000 or keys.dtype.kind not in 'iu':
        return np.argsort(keys, kind='stable')
    import torch
    return torch.sort(torch.from_numpy(keys.astype(np.int64, copy=False)), stable=True).indices.numpy()


def _unique_sorted(keys):
    """np.unique for large int64 arrays: torch's multi-threaded CPU sort is ~40x faster than numpy's at 4e7 keys."""
    keys = np.ascontiguousarray(keys, np.int64)
    if len(keys) < 1_000_000:
        return np.unique(keys)
    import torch
    srt = torch.sort(torch.from_numpy(keys)).values.numpy()
    return srt[np.concatenate(([True], srt[1:] != srt[:-1]))]


class InteractionData:
    def __init__(self, users, items, interactions, timestamp=None):
        self.user = np.asarray(users)
        self.item = np.asarray(items)
        self.interaction = np.asarray(interactions)
        assert len(self.user) == len(self.item) == len(self.interaction)
        self.timestamp = None if timestamp is None else np.asarray(timestamp)     # optional: orders Caser's sequences
        assert self.timestamp is None or len(self.timestamp) == len(self.user)
        self.has_internal_ids = False
        self.uid = self.iid = None
        self._users = self._items = None
        self._user_map = self._item_map = None
        self._cache = {}

    # ------------------------------------------------------------------ construction
    @classmethod
    def read_df(cls, df, user_label='user', item_label='item', interaction_label='interaction', timestamp_label=None,
                **kwds):
        ts = df[timestamp_label].values if timestamp_label is not None else None
        return cls(df[user_label].values, df[item_label].values, df[interaction_label].values, timestamp=ts)

    @classmethod
    def from_dataset(cls, ds):
        """Accepts an InteractionData or any object shaped like the reference's InteractionDataset."""
        if isinstance(ds, cls):
            return ds
        df = getattr(ds, '_df', None)
        if df is not None and all(c in df.columns for c in ('user', 'item', 'interaction')):
            ts = df['timestamp'].values if 'timestamp' in df.columns else None
            return cls(df['user'].values, df['item'].values, df['interaction'].values, timestamp=ts)
        if hasattr(ds, 'values_list'):
            rows = ds.values_list(['user', 'item', 'interaction'], to_list=True)
            u, i, v = zip(*rows) if rows else ((), (), ())
            return cls(np.array(u), np.array(i), np.array(v))
        raise TypeError(f'cannot read interactions from {type(ds)}')

    def __len__(self):
        return len(self.user)

    # ------------------------------------------------------------------ id abstraction (mem_dataset.py:309-330)
    def assign_internal_ids(self):
        if self.has_internal_ids:
            return
        ucodes, users = pd.factorize(self.user)          # codes in order of first appearance
        icodes, items = pd.factorize(self.item)
        self.uid = ucodes.astype(np.int32)
        self.iid = icodes.astype(np.int32)
        self._users = np.asarray(users)
        self._items = np.asarray(items)
        self._user_map = {k: i for i, k in enumerate(self._users.tolist())}
        self._item_map = {k: i for i, k in enumerate(self._items.tolist())}
        self.has_internal_ids = True
        self._cache.clear()

    def user_to_uid(self, user):
        return self._user_map.get(user.item() if isinstance(user, np.generic) else user)

    def item_to_iid(self, item):
        return self._item_map.get(item.item() if isinstance(item, np.generic) else item)

    def uid_to_user(self, uid):
        return self._users[uid].item() if 0 <= uid < len(self._users) else None

    def iid_to_item(self, iid):
        return self._items[iid].item() if 0 <= iid < len(self._items) else None

    def _id_lookup(self, which, ids):
        """Vectorised raw -> internal ids; unknown ids map to -1.  Non-negative integer ids in a compact range go
        through a direct table (one gather), anything else through a binary search in the sorted raw ids."""
        raw = self._items if which == 'items' else self._users
        ids = np.asarray(ids)
        key = 'lut_' + which
        if key not in self._cache:
            lut = None
            if raw.dtype.kind in 'iu' and len(raw) and raw.min() >= 0 and raw.max() <= max(1 << 24, 8 * len(raw)):
                lut = np.full(int(raw.max()) + 2, -1, np.int64)       # last slot: everything out of range
                lut[raw] = np.arange(len(raw))
            self._cache[key] = lut
            order = np.argsort(raw, kind='stable')
            self._cache['sorted_' + which] = (raw[order], order.astype(np.int64))
        lut = self._cache[key]
        if lut is not None and ids.dtype.kind in 'iu':
            top = len(lut) - 1
            safe = np.where((ids >= 0) & (ids < top), ids, top) if len(ids) else ids
            return lut[safe]
        s_, order = self._cache['sorted_' + which]
        if not len(s_):
            return np.full(len(ids), -1, np.int64)
        pos = np.clip(np.searchsorted(s_, ids), 0, len(s_) - 1)
        return np.where(s_[pos] == ids, order[pos], -1)

    def items_to_iids(self, items):
        """Vectorised raw -> internal item ids; unknown ids map to -1."""
        return self._id_lookup('items', items)

    def users_to_uids(self, users):
        """Vectorised raw -> internal user ids; unknown ids map to -1."""
        return self._id_lookup('users', users)

    @property
    def raw_items(self):
        return self._items

    @property
    def raw_users(self):
        return self._users

    def count_unique(self, column):
        if column in ('uid', 'user'):
            return len(self._users) if self.has_internal_ids else len(np.unique(self.user))
        if column in ('iid', 'item'):
            return len(self._items) if self.has_internal_ids else len(np.unique(self.item))
        raise ValueError(column)

    def min(self, column='interaction'):
        return getattr(self, column).min()

    def max(self, column='interaction'):
        return getattr(self, column).max()

    # ------------------------------------------------------------------ sparse views
    def csr(self, threshold=None):
        """(indptr int64, indices int32, data float64) over users x items; duplicates summed first, then entries
        with summed value < threshold dropped (cdae.py:61 binarises the summed row)."""
        key = ('csr', threshold)
        if key not in self._cache:
            assert self.has_internal_ids
            U, I = self.count_unique('uid'), self.count_unique('iid')
            indptr, indices, data = _build_csr(self.uid, self.iid, self.interaction, U, I)
            if threshold is not None:
                keep = data >= threshold
                rows = np.repeat(np.arange(U), np.diff(indptr))[keep]
                indices, data = indices[keep], data[keep]
                indptr = np.zeros(U + 1, np.int64)
                np.cumsum(np.bincount(rows, minlength=U), out=indptr[1:])
            self._cache[key] = (indptr, indices, data)
        return self._cache[key]

    def csc(self):
        if 'csc' not in self._cache:
            assert self.has_internal_ids
            U, I = self.count_unique('uid'), self.count_unique('iid')
            self._cache['csc'] = _build_csr(self.iid, self.uid, self.interaction, I, U)
        return self._cache['csc']

    def rows_by_user(self, threshold=None):
        """Per-user rows in DataFrame (insertion) order, filtered by interaction >= threshold
        (select_random_generator's view, mem_dataset.py:119-129)."""
        key = ('rows', threshold)
        if key not in self._cache:
            assert self.has_internal_ids
            U = self.count_unique('uid')
            sel = np.arange(len(self)) if threshold is None else np.flatnonzero(self.interaction >= threshold)
            order = sel[_argsort_stable(self.uid[sel])]
            indptr = np.zeros(U + 1, np.int64)
            np.cumsum(np.bincount(self.uid[sel], minlength=U), out=indptr[1:])
            self._cache[key] = (indptr, np.ascontiguousarray(self.iid[order]),
                                np.ascontiguousarray(self.interaction[order].astype(np.float64)))
        return self._cache[key]

    def select_user_interaction_vec(self, uid):
        from scipy.sparse import csr_matrix
        indptr, indices, data = self.csr()
        lo, hi = indptr[uid], indptr[uid + 1]
        return csr_matrix((data[lo:hi], indices[lo:hi], [0, hi - lo]), shape=(1, self.count_unique('iid')))

    def select_item_interaction_vec(self, iid):
        from scipy.sparse import csr_matrix
        indptr, indices, data = self.csc()
        lo, hi = indptr[iid], indptr[iid + 1]
        return csr_matrix((data[lo:hi], indices[lo:hi], [0, hi - lo]), shape=(1, self.count_unique('uid')))

    def user_items(self, uid):
        indptr, indices, _ = self.csr()
        return indices[indptr[uid]:indptr[uid + 1]]


def synthetic_interactions(n_users, n_items, nnz, seed=10, zipf_a=0.0, rating_low=1, rating_high=5):
    """Synthetic MovieLens-shaped data (SURVEY.md section 8d): unique (user, item) pairs, every user and item
    present, raw ids = internal id + 1, integer ratings uniform in [rating_low, rating_high], rows in random
    order.  zipf_a > 0 draws items from a Zipf-like popularity law (p_i ~ 1/(i+1)^a) and user activity
    log-normally, for the large configs."""
    rng = np.random.default_rng(seed)
    if zipf_a <= 0:
        total = n_users * n_items
        if total < 2 ** 62 and nnz <= total:
            pairs = rng.choice(total, nnz, replace=False) if total <= 50_000_000 else \
                np.unique(rng.integers(0, total, int(nnz * 1.05)))[:nnz]
            rng.shuffle(pairs)
        u, i = pairs // n_items, pairs % n_items
    else:
        act = rng.lognormal(0.0, 1.0, n_users)
        p_user = act / act.sum()
        pop = 1.0 / np.power(np.arange(1, n_items + 1, dtype=np.float64), zipf_a)
        cdf = np.cumsum(pop / pop.sum())
        key = np.zeros(0, np.int64)
        want, factor = nnz, 2.0
        for _ in range(8):       # duplicates of popular items are dropped: oversample, top up until nnz unique pairs exist
            deg = np.minimum(rng.multinomial(int(want * factor) + 16, p_user), n_items)
            uu = np.repeat(np.arange(n_users, dtype=np.int64), deg)
            ii = np.searchsorted(cdf, rng.random(len(uu))).clip(0, n_items - 1)
            new = _unique_sorted(uu * n_items + ii)
            key = new if not len(key) else _unique_sorted(np.concatenate([key, new]))
            want, factor = nnz - len(key), 4.0
            if want <= 0:
                break
        if len(key) > nnz:       # drop a random subset of the surplus
            drop = rng.choice(len(key), len(key) - nnz, replace=False)
            keep = np.ones(len(key), bool)
            keep[drop] = False
            key = key[keep]
        u, i = key // n_items, key % n_items
    # make sure every user / item id occurs so that the nominal shape is the actual shape
    miss_u = np.setdiff1d(np.arange(n_users), u)
    miss_i = np.setdiff1d(np.arange(n_items), i)
    if len(miss_u):
        u = np.concatenate([u, miss_u]); i = np.concatenate([i, rng.integers(0, n_items, len(miss_u))])
    if len(miss_i):
        i = np.concatenate([i, miss_i]); u = np.concatenate([u, rng.integers(0, n_users, len(miss_i))])
    key = _unique_sorted(u.astype(np.int64) * n_items + i)
    rng.shuffle(key)
    u, i = key // n_items, key % n_items
    val = rng.integers(rating_low, rating_high + 1, len(u))
    return (u + 1).astype(np.int64), (i + 1).astype(np.int64), val.astype(np.int64)


def synthetic_item_shard(n_users, n_items, nnz, rank, world, seed=10, zipf_a=1.0, device=None):
    """The columns [rank * ceil(n_items / world), ...) of a synthetic users x items interaction matrix with about `nnz`
    entries in total, generated WITHOUT ever forming the whole matrix (BASELINE.json configs[4]: 10 M x 1 M, 1 B
    interactions does not fit one process comfortably, and every rank only ever touches its own columns).
    Log-normal user activity (the same for every shard: seeded by `seed` alone), Zipf(zipf_a) item popularity inside the
    shard (stratified draws), unique (user, item) pairs, items sorted inside a user's row.  With device='cuda:k' the
    125 M entries of a configs[4] shard are drawn on the GPU in a fraction of a second and stay there.
    Returns (indptr int64 numpy [n_users + 1], indices int32 local item ids: numpy, or a torch tensor on `device`)."""
    import torch
    dev = torch.device(device) if device is not None else torch.device('cpu')
    per = -(-n_items // world)
    lo, hi = min(n_items, rank * per), min(n_items, (rank + 1) * per)
    n_loc = hi - lo
    act = np.random.default_rng(seed).lognormal(0.0, 1.0, n_users)
    lam = act * (nnz / world / act.sum())                       # expected entries of every user in this shard
    rng = np.random.default_rng(seed * 7919 + 1 + rank)
    deg = np.minimum(rng.poisson(lam), n_loc).astype(np.int64)
    total = int(deg.sum())
    # stratified draws: entry j of a row with d entries takes the popularity quantile (j + u) / d, so a row comes out
    # sorted without any sort; equal neighbours (several strata of an active user inside one popular item) are dropped
    g = torch.Generator(device=dev).manual_seed(seed * 104729 + rank)
    tdeg = torch.from_numpy(deg).to(dev)
    rows = torch.repeat_interleave(torch.arange(n_users, dtype=torch.int64, device=dev), tdeg)
    start = torch.cumsum(tdeg, 0) - tdeg
    q = torch.arange(total, dtype=torch.float64, device=dev) - start[rows].double()
    q += torch.rand(total, generator=g, dtype=torch.float64, device=dev)
    q /= tdeg[rows].double()
    if zipf_a > 0:
        pop = 1.0 / np.power(np.arange(1, n_loc + 1, dtype=np.float64), zipf_a)
        cdf = torch.from_numpy(np.cumsum(pop / pop.sum())).to(dev)
        items = torch.searchsorted(cdf, q).clamp_(0, n_loc - 1)
    else:
        items = (q * n_loc).long().clamp_(0, n_loc - 1)
    del q
    keep = torch.ones(total, dtype=torch.bool, device=dev)
    keep[1:] = (items[1:] != items[:-1]) | (rows[1:] != rows[:-1])
    rows, items = rows[keep], items[keep]
    indices = items.to(torch.int32)
    indptr = np.zeros(n_users + 1, np.int64)
    np.cumsum(torch.bincount(rows, minlength=n_users).cpu().numpy(), out=indptr[1:])
    return indptr, (indices if device is not None else indices.numpy())
