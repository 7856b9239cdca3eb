"""Dataset splits on the path into ranking_evaluation (SURVEY.md section 8f, rank 2): leave_k_out.

Mirrors DRecPy/Evaluation/Splits/leave_k_out.py:14-135 -- same signature, asserts, per-user generators
(random.Random(seed + idx + 1): the seed is incremented before each user's generator is created, :68-69) and row
selection (rng.sample over the user's rows in DataFrame order, :131-133) -- but for all users in one native call
(drb_leave_k_out, host C++ MT19937 replay, multi-threaded) instead of one `select('user == ...')` scan per user.
Returns two InteractionData objects whose rows keep the order of the input (InteractionDataset.drop semantics), with
the input's timestamps when it has them.
"""
import os
from heapq import heappush, heapreplace

import numpy as np
import pandas as pd

from . import _lib
from .dataset import InteractionData, _argsort_stable


def _group_rows_by_user(users):
    """Row positions grouped by user in order of first appearance, each group in row order."""
    codes, uniques = pd.factorize(np.asarray(users))
    order = _argsort_stable(codes)
    indptr = np.zeros(len(uniques) + 1, np.int64)
    np.cumsum(np.bincount(codes, minlength=len(uniques)), out=indptr[1:])
    return order.astype(np.int64), indptr


def leave_k_out(interaction_dataset, k=1, min_user_interactions=0, last_timestamps=False, timestamp_label='timestamp',
                seed=0, max_concurrent_threads=4, **kwds):
    assert k > 0, f'The value of k ({k}) must be > 0.'
    assert max_concurrent_threads > 0, f'The value of max_concurrent_threads ({max_concurrent_threads}) must be > 0.'
    ratio_variant = isinstance(k, float)
    if ratio_variant and k >= 1:
        raise Exception('The k parameter should be in the (0, 1) range when it\'s used as the percentage of '
                        'interactions to sample to the test set, per user. Current value: ' + str(k))
    timestamps = kwds.get('timestamps')
    if timestamps is None and last_timestamps:
        df = getattr(interaction_dataset, '_df', None)
        if df is not None and timestamp_label in getattr(df, 'columns', ()):
            timestamps = df[timestamp_label].values
        else:
            timestamps = getattr(interaction_dataset, timestamp_label, None)
        assert timestamps is not None, f'No "{timestamp_label}" values to split by (pass timestamps=...)'
    ds = InteractionData.from_dataset(interaction_dataset)
    order, indptr = _group_rows_by_user(ds.user)
    n_users = len(indptr) - 1
    flags = np.zeros(len(ds), np.uint8)          # per grouped position: 0 train, 1 test, 2 removed
    if not last_timestamps:
        _lib.check(_lib.load().drb_leave_k_out(
            n_users, _lib.np_ptr(indptr), 0 if ratio_variant else int(k), float(k) if ratio_variant else 0.0,
            int(ratio_variant), int(min_user_interactions), int(seed), min(max(int(max_concurrent_threads), 1), 64),
            _lib.np_ptr(flags)))
    else:
        # leave_k_out.py:120-126: a k-sized heap of (timestamp, rid) fed in row order; once full every further row
        # *replaces* the current minimum (heapreplace, whether or not it is newer) -- kept as is
        ts = np.asarray(timestamps)[order]
        for u in range(n_users):
            lo, hi = int(indptr[u]), int(indptr[u + 1])
            n = hi - lo
            ku = int(n * k) if ratio_variant else k
            if n < min_user_interactions:
                flags[lo:hi] = 2
            elif n > ku > 0:
                heap = []
                for pos in range(lo, hi):
                    entry = (ts[pos].item() if hasattr(ts[pos], 'item') else ts[pos], int(order[pos]), pos)
                    if len(heap) < ku: heappush(heap, entry)
                    else: heapreplace(heap, entry)
                for _, _, pos in heap:
                    flags[pos] = 1
    row_flag = np.empty(len(ds), np.uint8)
    row_flag[order] = flags
    tr, te = np.flatnonzero(row_flag == 0), np.flatnonzero(row_flag == 1)
    ts = ds.timestamp if ds.timestamp is not None else (None if timestamps is None else np.asarray(timestamps))
    return (InteractionData(ds.user[tr], ds.item[tr], ds.interaction[tr], None if ts is None else ts[tr]),
            InteractionData(ds.user[te], ds.item[te], ds.interaction[te], None if ts is None else ts[te]))
