"""ranking_evaluation with batched native scoring, and the ranking metrics on the path.

Mirrors DRecPy/Evaluation/Processes/ranking_evaluation.py:19-246 (same signature, asserts, per-user
random.Random(seed + idx) candidate generation, shuffle, model.rank, relevancies, round(sum / count, 4)) and
DRecPy/Evaluation/Metrics/ranking.py (DCG :20-56, NDCG :59-91, HitRatio :94-114, Recall, Precision).
What changes: the per-user candidate generation runs in libdrb's host C++ (drb_eval_candidates) and all users
are scored in one batched GPU call (model.rank_batch) instead of 4 Python threads calling model.rank per user.
Models without rank_batch (any object with .rank) and non-integer raw ids go through the same protocol in Python.

recommendation_evaluation (DRecPy/Evaluation/Processes/recommendation_evaluation.py:18-192, restated: see its
docstring) evaluates the full-catalog top-k of every test user; for CDAE / DMF the lists stay on the device and
drb_eval_topk_metrics reduces them to per-user DCG / ideal DCG / hit counts there.

predictive_evaluation (DRecPy/Evaluation/Processes/predictive_evaluation.py:7-65 with Metrics/regression.py, restated:
see its docstring) computes RMSE / MSE / MAE of model.predict over the test rows; CDAE and DMF score all rows in one
predict_batch call (drb_cdae_predict_pairs / drb_dmf_predict_pairs).
"""
import math
import os
import random
import time

import numpy as np
import pandas as pd

from . import _lib
from .dataset import InteractionData


# ------------------------------------------------------------------------------------------ metrics
class RankingMetricABC:
    @property
    def name(self):
        return self.__class__.__name__


class DCG(RankingMetricABC):
    def __init__(self, strong_relevancy=True):
        self.strong_relevancy = strong_relevancy

    def __call__(self, recommendations, k=None, relevancies=None):
        if relevancies is None: return 0
        if k is not None: recommendations = recommendations[:k]
        curr_dcg = 0
        for i, r in enumerate(recommendations):
            rel = float(relevancies[r])
            if self.strong_relevancy:
                curr_dcg += (2 ** rel - 1) / math.log2(2 + i)
            else:
                curr_dcg += rel / math.log2(2 + i)
        return curr_dcg


class NDCG(RankingMetricABC):
    def __init__(self, strong_relevancy=True):
        self.strong_relevancy = strong_relevancy
        self.dcg = DCG(strong_relevancy=strong_relevancy)

    def __call__(self, recommendations, k=None, relevancies=None):
        if relevancies is None: return 0
        curr_dcg = self.dcg(recommendations, relevancies=relevancies, k=k)
        best_recommendations = sorted(relevancies.keys(), key=lambda x: -relevancies[x])
        best_dcg = self.dcg(best_recommendations, relevancies=relevancies, k=k)
        return curr_dcg / best_dcg


class HitRatio(RankingMetricABC):
    def __call__(self, recommendations, k=None, relevant_recommendations=None):
        if relevant_recommendations is None: return 0
        if k is not None: recommendations = recommendations[:k]
        recommendations = set([str(item) for item in recommendations])
        relevant_recommendations = set([str(item) for item in relevant_recommendations])
        return len(recommendations.intersection(relevant_recommendations)) / len(relevant_recommendations)


class Recall(RankingMetricABC):
    def __call__(self, recommendations, k=None, relevant_recommendations=None):
        if relevant_recommendations is None: return 0
        if k is not None: recommendations = recommendations[:k]
        in_common = set(recommendations).intersection(set(relevant_recommendations))
        return len(in_common) / len(relevant_recommendations)


class Precision(RankingMetricABC):
    def __call__(self, recommendations, k=None, relevant_recommendations=None):
        if relevant_recommendations is None: return 0
        if k is not None: recommendations = recommendations[:k]
        in_common = set(recommendations).intersection(set(relevant_recommendations))
        return len(in_common) / len(recommendations)


# ------------------------------------------------------------------------------------------ candidate generation
def _group_by_user(data):
    """unique users in first-appearance order + test rows grouped by user with row order preserved."""
    codes, users = pd.factorize(data.user)
    order = np.argsort(codes, kind='stable')
    indptr = np.zeros(len(users) + 1, np.int64)
    np.cumsum(np.bincount(codes, minlength=len(users)), out=indptr[1:])
    return np.asarray(users), indptr, order


def _train_positive_items(model, users, thr):
    """What drb_eval_candidates needs to test `raw item in training positives of user` without copying anything:
    the training CSR of positives over internal ids, the training row of every evaluated user, and the sorted
    raw-item -> internal-id map (ranking_evaluation.py:196-199)."""
    data = model._data if hasattr(model, '_data') else InteractionData.from_dataset(model.interaction_dataset)
    data.assign_internal_ids()
    indptr, indices, _ = data.csr(thr)
    rows = np.ascontiguousarray(data.users_to_uids(users).astype(np.int64))
    data.items_to_iids(np.zeros(0, np.int64))          # builds the cached sorted map
    raw_sorted, order = data._cache['sorted_items']
    return (rows, np.ascontiguousarray(indptr), np.ascontiguousarray(indices),
            np.ascontiguousarray(raw_sorted.astype(np.int64)), np.ascontiguousarray(order.astype(np.int32)))


def generate_candidates(model, data, users, t_indptr, t_order, thr, n_pos, n_neg, generate_negative_pairs,
                        train_evaluation, seed):
    """ranking_evaluation.py:163-219 for every user at once (native).  Returns cand_off, cand, pos_off, pos,
    skipped."""
    n_users = len(users)
    t_item = np.ascontiguousarray(data.item[t_order].astype(np.int64))
    t_val = np.ascontiguousarray(data.interaction[t_order].astype(np.float64))
    black = None
    if not train_evaluation and generate_negative_pairs:
        black = _train_positive_items(model, users, thr)
    is_frac = isinstance(n_neg, float)
    per_user_neg = 0 if n_neg is None else (int(np.ceil(n_neg * np.diff(t_indptr).max())) if is_frac else int(n_neg))
    cap = int(len(t_item) + n_users * per_user_neg + 16)
    cand_off = np.zeros(n_users + 1, np.int64)
    pos_off = np.zeros(n_users + 1, np.int64)
    cand = np.empty(cap, np.int64)
    pos = np.empty(cap, np.int64)
    skipped = np.zeros(n_users, np.uint8)
    bp = [_lib.np_ptr(a) for a in black] if black is not None else [None] * 5
    _lib.check(_lib.load().drb_eval_candidates(
        n_users, _lib.np_ptr(t_indptr), _lib.np_ptr(t_item), _lib.np_ptr(t_val), bp[0], bp[1], bp[2], bp[3], bp[4],
        len(black[3]) if black is not None else 0, int(bool(train_evaluation)), int(model.n_items), float(thr),
        -1 if n_pos is None else int(n_pos), -1.0 if n_neg is None else float(n_neg), int(is_frac),
        int(bool(generate_negative_pairs)), int(seed), min(16, os.cpu_count() or 1), cap, _lib.np_ptr(cand_off),
        _lib.np_ptr(cand), _lib.np_ptr(pos_off), _lib.np_ptr(pos), _lib.np_ptr(skipped)))
    return cand_off, cand[:cand_off[-1]], pos_off, pos[:pos_off[-1]], skipped, t_item, t_val


def _candidates_python(rng, test_rows, train_pos_items, test_pos_items, n_items, thr, n_pos, n_neg, generate,
                       train_evaluation):
    """The same protocol in Python (non-integer raw ids)."""
    pos = [(it, v) for it, v in test_rows if v >= thr]
    if n_pos is None:
        chosen = pos
    else:
        if len(pos) < n_pos: return None
        chosen = rng.sample(pos, n_pos)
    positives = [it for it, _ in chosen]
    neg_pool = [it for it, v in test_rows if v < thr]
    if n_neg is None:
        negatives = list(neg_pool)
    else:
        if isinstance(n_neg, float): n_neg = int(n_neg * len(positives))
        negatives = rng.sample(neg_pool, min(n_neg, len(neg_pool)))
        if len(negatives) < n_neg and generate:
            blacklist = set(test_pos_items) if train_evaluation else set(train_pos_items) | set(test_pos_items)
            if n_items - len(blacklist) < n_neg: return None
            while len(negatives) < n_neg:
                new_item = rng.randint(0, n_items - 1)
                if new_item not in blacklist and new_item not in negatives:
                    negatives.append(new_item)
    all_items = positives + negatives
    if len(all_items) == 0: return None
    rng.shuffle(all_items)
    return all_items, positives


# ------------------------------------------------------------------------------------------ vectorised protocol
def _fast_evaluation(model, data, users, t_indptr, t_order, thr, n_pos, n_neg, generate, train_evaluation, seed,
                     novelty, metrics, ks):
    """Same protocol as the per-user loop below for the built-in metrics, with every per-user Python step replaced
    by array operations that perform the SAME float64 operations in the SAME order per user (sequential DCG sums,
    sequential sum over users), so the rounded results are identical.  Returns None when a corner case needs the
    general path (duplicate items inside one user's candidate / positive list)."""
    cand_off, cand, pos_off, pos, skipped, t_item, t_val = generate_candidates(
        model, data, users, t_indptr, t_order, thr, n_pos, n_neg, generate, train_evaluation, seed)
    active = np.flatnonzero(skipped == 0)
    t_item, t_val = t_item[:t_indptr[-1]], t_val[:t_indptr[-1]]    # rows of the evaluated users only
    metric_sums = {(m.name, k_): [0, 0] for m in metrics for k_ in ks}
    if len(active):
        known = model._data.users_to_uids(users[active]) >= 0       # model.rank asserts the user is known -> skipped
        active = active[known]
    if len(active):
        n = len(active)
        c_lens = (cand_off[active + 1] - cand_off[active]).astype(np.int64)
        p_lens = (pos_off[active + 1] - pos_off[active]).astype(np.int64)
        c_off = np.zeros(n + 1, np.int64); np.cumsum(c_lens, out=c_off[1:])
        p_off = np.zeros(n + 1, np.int64); np.cumsum(p_lens, out=p_off[1:])
        # equal list lengths (the usual protocol: n_pos positives + n_neg negatives for everybody) need no per-element
        # segment arithmetic: the source index is a broadcast add, the relevancy matrix a reshape
        uniform_c = int(c_lens.min()) == int(c_lens.max())
        uniform_p = int(p_lens.min()) == int(p_lens.max())
        c_seg = p_seg = None

        def flatten(off, flat, lens, tot, uniform):
            """The active users' lists back to back (+ the segment ids when the lengths differ)."""
            if uniform and len(flat) >= tot and off[active[0]] == 0 and off[active[-1] + 1] == tot:
                return flat[:tot], None        # every list in between is empty: they already lie back to back
            if uniform:
                return flat[(off[active][:, None] + np.arange(int(lens[0]), dtype=np.int64)[None, :]).ravel()], None
            seg = np.repeat(np.arange(n), lens)
            start = np.zeros(n, np.int64); np.cumsum(lens[:-1], out=start[1:])
            return flat[np.arange(tot) - np.repeat(start, lens) + np.repeat(off[active], lens)], seg
        c_flat, c_seg = flatten(cand_off, cand, c_lens, int(c_off[-1]), uniform_c)
        p_flat, p_seg = flatten(pos_off, pos, p_lens, int(p_off[-1]), uniform_p)
        big = int(max(c_flat.max(initial=0), t_item.max(initial=0), p_flat.max(initial=0))) + 2
        if big * (len(users) + 1) >= 2 ** 62 or c_flat.min(initial=0) < 0 or t_item.min(initial=0) < 0:
            return None
        # corner case: duplicate items inside one candidate or positive list -> general path.  Positives and negatives
        # are distinct test rows of the user and generated negatives avoid both (ranking_evaluation.py:163-219), so a
        # list can only repeat an item when the user's test rows do: check those (one key per test row) first.
        t_seg = np.repeat(np.arange(len(users)), np.diff(t_indptr))
        tk = np.sort(t_seg * big + t_item)
        if len(tk) > 1 and (tk[1:] == tk[:-1]).any():
            if c_seg is None: c_seg = np.repeat(np.arange(n), c_lens)
            if p_seg is None: p_seg = np.repeat(np.arange(n), p_lens)
            ck = np.sort(c_seg * big + c_flat)
            pk = np.sort(p_seg * big + p_flat)
            if (len(ck) > 1 and (ck[1:] == ck[:-1]).any()) or (len(pk) > 1 and (pk[1:] == pk[:-1]).any()):
                return None
        ranked, n_out = model.rank_arrays(users[active], c_flat, c_off, novelty=novelty)
        L = ranked.shape[1]
        # per-user DCG / ideal DCG / hit counts at every cut-off, natively for all users (drb_eval_metrics: the relevancy
        # of an item is its first test row of the user, else 0 -- ranking_evaluation.py:223 --, a hit is a ranked item
        # among the user's sampled positives); same float64 operations in the same order as the metric classes above
        lib, nthr = _lib.load(), min(16, os.cpu_count() or 1)
        t_beg = np.ascontiguousarray(t_indptr[:-1][active].astype(np.int64))
        t_end = np.ascontiguousarray(t_indptr[1:][active].astype(np.int64))
        t_item_c, t_val_c = np.ascontiguousarray(t_item, np.int64), np.ascontiguousarray(t_val, np.float64)
        ranked_c = np.ascontiguousarray(ranked, np.int64)
        n_out_c = np.ascontiguousarray(n_out, np.int32)
        c_flat_c, p_flat_c = np.ascontiguousarray(c_flat, np.int64), np.ascontiguousarray(p_flat, np.int64)
        ks_c = np.ascontiguousarray(ks, np.int64)
        dcg, idcg = np.zeros((n, len(ks))), np.zeros((n, len(ks)))
        hits_all = np.zeros((n, len(ks)), np.int64)
        _lib.check(lib.drb_eval_metrics(
            n, _lib.np_ptr(t_beg), _lib.np_ptr(t_end), _lib.np_ptr(t_item_c), _lib.np_ptr(t_val_c), _lib.np_ptr(ranked_c),
            L, _lib.np_ptr(n_out_c), _lib.np_ptr(np.ascontiguousarray(c_off[:-1])), _lib.np_ptr(np.ascontiguousarray(c_off[1:])),
            _lib.np_ptr(c_flat_c), _lib.np_ptr(np.ascontiguousarray(p_off[:-1])), _lib.np_ptr(np.ascontiguousarray(p_off[1:])),
            _lib.np_ptr(p_flat_c), _lib.np_ptr(ks_c), len(ks), nthr, _lib.np_ptr(dcg), _lib.np_ptr(idcg),
            _lib.np_ptr(hits_all)))
        n_rec = np.minimum(np.asarray(n_out)[:, None], np.asarray(ks)[None, :])
        _metric_sums_from_user_values(metric_sums, metrics, ks, dcg, idcg, hits_all, n_rec, p_lens, p_lens)
    return _metric_results(metric_sums)


def _metric_sums_from_user_values(metric_sums, metrics, ks, dcg, idcg, hits_all, n_rec, n_pos, n_pos_distinct):
    """The built-in metrics of every evaluated user from its per-cut-off sums ([n_users, len(ks)] arrays: DCG, ideal DCG,
    hits among the first n_rec recommendations), added left to right in user order into metric_sums -- the same float
    operations in the same order as the per-user metric calls.  n_pos: length of the sampled positives list (Recall);
    n_pos_distinct: its distinct items (HitRatio divides by the size of a set).  A user whose metric would divide by
    zero is skipped for that (metric, k), as the per-user loop skips a metric that raises."""
    for m in metrics:
        for j, k_ in enumerate(ks):
            if type(m) is NDCG:
                cur, best = dcg[:, j], idcg[:, j]
                good = best != 0                                    # ZeroDivisionError -> metric skipped for the user
                vals = (cur[good] / best[good]).tolist()
            else:
                hits = hits_all[:, j]
                if type(m) is Precision:
                    good = n_rec[:, j] > 0
                    vals = (hits[good] / n_rec[good, j]).tolist()
                else:                                               # HitRatio, Recall: / number of positives
                    den = n_pos_distinct if type(m) is HitRatio else n_pos
                    good = den > 0
                    vals = (hits[good] / den[good]).tolist()
            acc = 0
            for v in vals:                                          # same left-to-right float additions as the loop
                acc += v
            metric_sums[(m.name, k_)] = [acc, len(vals)]


def _metric_results(metric_sums):
    return {m + f'@{k_}': round(metric_sums[(m, k_)][0] / metric_sums[(m, k_)][1], 4)
            if metric_sums[(m, k_)][1] > 0 else 0 for m, k_ in metric_sums}


def _call_metrics(metric_sums, metrics, ks, recommendations, positives, best_item, relevancies):
    """ranking_evaluation.py:223-246: every metric gets the arguments its __call__ names; an exception skips that
    (metric, k) for the user."""
    for m in metrics:
        param_names = m.__call__.__code__.co_varnames
        for k_ in ks:
            params = dict()
            for param_name in param_names:
                if param_name == 'recommendations': params[param_name] = recommendations
                elif param_name == 'relevant_recommendations': params[param_name] = positives
                elif param_name == 'relevant_recommendation': params[param_name] = best_item
                elif param_name == 'relevancies': params[param_name] = relevancies
                elif param_name == 'k': params[param_name] = k_
            try:
                metric_sums[(m.name, k_)][0] += m(**params)
                metric_sums[(m.name, k_)][1] += 1
            except Exception:
                pass


# ------------------------------------------------------------------------------------------ the protocol
def ranking_evaluation(model, ds_test=None, n_test_users=None, k=10, n_pos_interactions=None, n_neg_interactions=None,
                       generate_negative_pairs=False, novelty=False, seed=0, max_concurrent_threads=4, **kwds):
    assert n_test_users is None or n_test_users > 0, f'The number of test users ({n_test_users}) should be > 0.'
    assert n_pos_interactions is None or n_pos_interactions > 0, \
        f'The number of positive interactions ({n_pos_interactions}) should be None or an integer > 0.'
    assert n_neg_interactions is None or n_neg_interactions > 0, \
        f'The number of negative interactions ({n_neg_interactions}) should be None or an integer > 0.'
    if generate_negative_pairs and n_neg_interactions is None:
        raise Exception('Cannot generate negative interaction pairs when the number of negative interactions per user '
                        'is not defined. Either set generate_negative_pairs=False or define the n_neg_interactions '
                        'parameter.')
    interaction_threshold = kwds.get('interaction_threshold', model.interaction_threshold)
    if type(k) is not list: k = [k]
    for k_ in k: assert k_ > 0, f'k ({k_}) should be > 0.'

    train_evaluation = False
    if ds_test is None or ds_test is model.interaction_dataset or ds_test is getattr(model, '_data', None):
        train_evaluation = True
        ds_test = model.interaction_dataset
    metrics = kwds.get('metrics', [Precision(), Recall(), HitRatio(), NDCG()])
    assert isinstance(metrics, list), f'Expected "metrics" argument to be a list and found {type(metrics)}. ' \
        f'Should contain instances of RankingMetricABC.'
    for m in metrics:
        assert hasattr(m, 'name') and callable(m), f'Expected metric {m} to be an instance of type RankingMetricABC.'

    data = InteractionData.from_dataset(ds_test)
    users, t_indptr, t_order = _group_by_user(data)
    n_eval = len(users) if n_test_users is None else min(n_test_users, len(users))
    users, t_indptr = users[:n_eval], np.ascontiguousarray(t_indptr[:n_eval + 1])
    metric_sums = {(m.name, k_): [0, 0] for m in metrics for k_ in k}
    record = kwds.get('record', None)      # optional list collecting (user, candidates, ranked) for tests

    native_ids = np.issubdtype(data.item.dtype, np.integer)
    fast = (native_ids and hasattr(model, 'rank_arrays') and record is None and not kwds.get('force_python', False)
            and all(type(m) in (HitRatio, NDCG, Precision, Recall) and getattr(m, 'strong_relevancy', True)
                    for m in metrics))
    if fast:
        res = _fast_evaluation(model, data, users, t_indptr, t_order, interaction_threshold, n_pos_interactions,
                               n_neg_interactions, generate_negative_pairs, train_evaluation, seed, novelty, metrics, k)
        if res is not None:
            return res
    if native_ids:
        cand_off, cand, pos_off, pos, skipped, t_item, t_val = generate_candidates(
            model, data, users, t_indptr, t_order, interaction_threshold, n_pos_interactions, n_neg_interactions,
            generate_negative_pairs, train_evaluation, seed)
        active = np.flatnonzero(skipped == 0)
        if len(active) and hasattr(model, '_data'):
            # model.rank asserts the user is known; the reference logs that failure and skips the user
            # (ranking_evaluation.py:222 inside the per-user try) -- same filter as the vectorised path
            active = active[model._data.users_to_uids(users[active]) >= 0]
        cand_lists = [cand[cand_off[u]:cand_off[u + 1]] for u in active]
        pos_lists = [pos[pos_off[u]:pos_off[u + 1]].tolist() for u in active]
        rows = [(t_item[t_indptr[u]:t_indptr[u + 1]], t_val[t_indptr[u]:t_indptr[u + 1]]) for u in active]
    else:
        active, cand_lists, pos_lists, rows = [], [], [], []
        tr = InteractionData.from_dataset(model.interaction_dataset)
        for idx in range(n_eval):
            sl = t_order[t_indptr[idx]:t_indptr[idx + 1]]
            trows = list(zip(data.item[sl].tolist(), data.interaction[sl].tolist()))
            tpos = [it for it, v in trows if v >= interaction_threshold]
            sel = (tr.user == users[idx]) & (tr.interaction >= interaction_threshold)
            res = _candidates_python(random.Random(seed + idx), trows, tr.item[sel].tolist(), tpos, model.n_items,
                                     interaction_threshold, n_pos_interactions, n_neg_interactions,
                                     generate_negative_pairs, train_evaluation)
            if res is None: continue
            active.append(idx)
            cand_lists.append(np.asarray(res[0], dtype=object))
            pos_lists.append(res[1])
            rows.append((data.item[sl], data.interaction[sl]))

    # ---- rank: one batched call when the model supports it (model.rank semantics, ranking_evaluation.py:222)
    if len(active) == 0:
        ranked_lists = []
    elif hasattr(model, 'rank_batch') and native_ids:
        ranked_lists = []
        chunk = kwds.get('rank_chunk', 16384)
        for o in range(0, len(active), chunk):
            sub_users = users[active[o:o + chunk]].tolist()
            rl, _, _ = model.rank_batch(sub_users, cand_lists[o:o + chunk], novelty=novelty)
            ranked_lists.extend(rl)
    else:
        ranked_lists = [[item for _, item in model.rank(users[u].item() if hasattr(users[u], 'item') else users[u],
                                                         list(c.tolist()), novelty=novelty, skip_invalid_items=True)]
                        for u, c in zip(active, cand_lists)]

    # ---- metrics (ranking_evaluation.py:223-246); exceptions inside a metric skip that (metric, k) for the user
    for u, all_items, positives, (r_items, r_vals), recommendations in zip(active, cand_lists, pos_lists, rows,
                                                                          ranked_lists):
        all_items = all_items.tolist()
        first_val = {}
        for it, v in zip(r_items.tolist(), r_vals.tolist()):
            first_val.setdefault(it, v)
        relevancies = {item: (first_val.get(item) or 0) for item in all_items}
        best_item = None if len(positives) == 0 else min(positives, key=lambda it: relevancies[it])
        if record is not None:
            record.append((users[u].item() if hasattr(users[u], 'item') else users[u], all_items, list(recommendations)))
        _call_metrics(metric_sums, metrics, k, recommendations, positives, best_item, relevancies)

    return _metric_results(metric_sums)


# ------------------------------------------------------------------------------------------ recommendation_evaluation
_TOPK_MAX = 2048            # longest list the models' full-catalog top-k (topk_batch) produces


def _float32_from_order(o):
    """Inverse of the order-preserving map float32 -> uint32 (the f2ord of the top-k kernels)."""
    u = (o & 0x7fffffff) if o & 0x80000000 else (~o & 0xffffffff)
    return np.array([u], np.uint32).view(np.float32)


def _score_cut(model, threshold):
    """recommend(..., interaction_threshold=t) keeps an item when its reported score is >= t.  The reported score is a
    non-decreasing function of the float32 top-k score (CDAE: the score itself, so NumPy compares in float32; DMF: the
    rescaled p, in float64 when the interaction bounds are NumPy scalars), so the kept items are those whose top-k score
    is >= the smallest finite float32 whose reported score passes.  Found by bisection over the float32 values in
    order, with the same NumPy comparison recommend() makes.  NaN when no finite float32 passes (no score is >= NaN)."""
    def keeps(o):
        with np.errstate(all='ignore'):
            return bool(model._reported_scores(_float32_from_order(o))[0] >= threshold)
    lo, hi = 0x00800000, 0xff7fffff             # order keys of -FLT_MAX and FLT_MAX
    if not keeps(hi):
        return float('nan')
    while lo < hi:
        mid = (lo + hi) // 2
        if keeps(mid): hi = mid
        else: lo = mid + 1
    return float(_float32_from_order(lo)[0])


def _fast_recommendation_evaluation(model, data, users, t_indptr, t_order, thr, n_pos, train_evaluation, seed, novelty,
                                    low_threshold, metrics, ks, chunk, timings):
    """The protocol of the per-user loop in recommendation_evaluation for the built-in metrics, with the top-k lists
    and the per-user metric sums on the device.  Returns None when a corner case needs the general path (a negative
    relevancy: the reference's ideal list then ranks the recommended items outside the evaluated set, which count 0,
    above it)."""
    import torch
    t0 = time.perf_counter()
    cand_off, cand, pos_off, pos, skipped, t_item, t_val = generate_candidates(
        model, data, users, t_indptr, t_order, thr, n_pos, None, False, train_evaluation, seed)
    metric_sums = {(m.name, k_): [0, 0] for m in metrics for k_ in ks}
    active = np.flatnonzero(skipped == 0)
    if len(active):
        active = active[model._data.users_to_uids(users[active]) >= 0]     # recommend() asserts -> user skipped
    n = len(active)
    if n == 0:
        return _metric_results(metric_sums)
    t_item, t_val = t_item[:t_indptr[-1]], t_val[:t_indptr[-1]]

    # every (user, item) pair as one integer key: the user's evaluation index and the item's code among the test items
    codes, uniq = pd.factorize(t_item)
    nc = max(len(uniq), 1)
    code_index = pd.Index(uniq)
    tkey = np.repeat(np.arange(len(users), dtype=np.int64), np.diff(t_indptr)) * nc + codes
    srt = np.argsort(tkey, kind='stable')               # rows of one key stay in row order: the first comes first
    tk = tkey[srt]
    first = np.concatenate(([True], tk[1:] != tk[:-1]))
    tkey_first, tval_first = tk[first], t_val[srt][first]

    def members(off, flat):
        """The active users' lists back to back: (items, evaluation index of their user, list lengths)."""
        lens = (off[active + 1] - off[active]).astype(np.int64)
        start = np.zeros(n, np.int64)
        np.cumsum(lens[:-1], out=start[1:])
        idx = np.arange(int(lens.sum()), dtype=np.int64) - np.repeat(start - off[active], lens)
        return flat[idx], np.repeat(active.astype(np.int64), lens), lens
    c_items, c_user, _ = members(cand_off, cand)
    p_items, p_user, p_lens = members(pos_off, pos)
    ekey = np.unique(c_user * nc + code_index.get_indexer(c_items))     # distinct items of every evaluated set C
    pkey = np.unique(p_user * nc + code_index.get_indexer(p_items))     # distinct sampled positives
    e_val = tval_first[np.searchsorted(tkey_first, ekey)]               # value of the user's first test row
    if not (e_val >= 0).all():
        return None
    j = np.minimum(np.searchsorted(pkey, ekey), max(len(pkey) - 1, 0))
    e_pos = (pkey[j] == ekey) if len(pkey) else np.zeros(len(ekey), bool)
    e_row = np.searchsorted(active, ekey // nc)                         # row of the user among the active users
    p_distinct = np.bincount(np.searchsorted(active, pkey // nc), minlength=n).astype(np.int64)
    # gains 2 ** rel - 1 as the metric classes compute them (C library pow), once per distinct value
    vals, inv = np.unique(e_val, return_inverse=True)
    e_gain = np.array([2 ** float(v) - 1 for v in vals.tolist()], np.float64)[inv.ravel()]
    ideal_off = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(e_row, minlength=n), out=ideal_off[1:])      # ekey is sorted by user: rows are contiguous
    e_iid = np.asarray(model._data.items_to_iids(uniq[ekey % nc]), np.int64)
    known = np.flatnonzero(e_iid >= 0)                                  # items the model can recommend
    lut = known[np.argsort(e_row[known] * (int(model.n_items) + 1) + e_iid[known], kind='stable')]   # by (user, iid)
    lut_off = np.zeros(n + 1, np.int64)
    np.cumsum(np.bincount(e_row[lut], minlength=n), out=lut_off[1:])
    K = max(ks)
    disc = np.array([math.log2(2 + i) for i in range(K)], np.float64)
    use_thr = low_threshold is not None
    cut = _score_cut(model, low_threshold) if use_thr else 0.0
    uids = np.asarray(model._data.users_to_uids(users[active]), np.int32)
    t1 = time.perf_counter()

    dev = model._dev

    def up(a, dtype):
        a = np.ascontiguousarray(a, dtype)
        return torch.from_numpy(a if len(a) else np.zeros(1, dtype)).to(dev)   # never a NULL device pointer
    d = {'uids': up(uids, np.int32), 'lut_off': up(lut_off, np.int64), 'lut_iid': up(e_iid[lut], np.int32),
         'lut_gain': up(e_gain[lut], np.float64), 'lut_pos': up(e_pos[lut], np.uint8),
         'ideal_off': up(ideal_off, np.int64), 'ideal_gain': up(e_gain, np.float64), 'disc': up(disc, np.float64),
         'ks': up(ks, np.int32)}
    nk = len(ks)
    d_dcg = torch.empty((n, nk), dtype=torch.float64, device=dev)
    d_idcg = torch.empty((n, nk), dtype=torch.float64, device=dev)
    d_hits = torch.empty((n, nk), dtype=torch.int32, device=dev)
    d_nrec = torch.empty((n, nk), dtype=torch.int32, device=dev)
    lib, P = _lib.load(), _lib.t_ptr
    ev = [] if timings is not None else None
    with model._lock:
        stream = model._stream                          # the stream libdrb enqueues on
        for o in range(0, n, chunk):
            c = min(chunk, n - o)
            if ev is not None:
                ev.append([torch.cuda.Event(enable_timing=True) for _ in range(3)])
                ev[-1][0].record(stream)
            o_i, o_s, o_n = model._topk_device_scores(d['uids'][o:o + c], K, novelty)
            if ev is not None:
                ev[-1][1].record(stream)
            _lib.check(lib.drb_eval_topk_metrics(
                model._ctx, c, P(o_i), P(o_s), K, P(o_n), int(use_thr), cut, P(d['lut_off'][o:]), P(d['lut_iid']),
                P(d['lut_gain']), P(d['lut_pos']), P(d['ideal_off'][o:]), P(d['ideal_gain']), P(d['disc']), P(d['ks']),
                nk, K, P(d_dcg[o:]), P(d_idcg[o:]), P(d_hits[o:]), P(d_nrec[o:])))
            if ev is not None:
                ev[-1][2].record(stream)
        t2 = time.perf_counter()
        dcg, idcg = d_dcg.cpu().numpy(), d_idcg.cpu().numpy()
        hits, n_rec = d_hits.cpu().numpy(), d_nrec.cpu().numpy()
    t3 = time.perf_counter()
    _metric_sums_from_user_values(metric_sums, metrics, ks, dcg, idcg, hits, n_rec, p_lens, p_distinct)
    res = _metric_results(metric_sums)
    if timings is not None:
        timings.update(host_protocol_s=(t1 - t0) + (time.perf_counter() - t3), launch_and_upload_s=t2 - t1,
                       copy_back_s=t3 - t2, topk_ms=sum(a.elapsed_time(b) for a, b, _ in ev),
                       metrics_kernel_ms=sum(b.elapsed_time(c_) for _, b, c_ in ev), n_users=n,
                       per_user={'dcg': dcg, 'idcg': idcg, 'hits': hits, 'n_rec': n_rec, 'users': users[active]})
    return res


def recommendation_evaluation(model, ds_test=None, n_test_users=None, k=10, n_pos_interactions=None, novelty=False,
                              ignore_low_predictions_threshold=None, metrics=None, max_concurrent_threads=4, seed=0,
                              verbose=True, **kwds):
    """Full-catalog recommendation metrics of every test user (DRecPy's recommendation_evaluation protocol, same
    signature).  Returns {'<metric>@<k>': value}.

    Test users are taken in order of first appearance in ds_test (the first n_test_users of them).  For test user idx:
      1. rng = random.Random(seed + idx);
      2. positives: the user's test rows, in row order, with value >= interaction_threshold (the model's, or the
         `interaction_threshold` keyword); all of them if n_pos_interactions is None, else rng.sample(positives,
         n_pos_interactions), and a user with fewer positives than that is skipped;
      3. the evaluated set C: the sampled positives plus every test row of the user below the threshold (what
         ranking_evaluation evaluates with n_neg_interactions=None, generate_negative_pairs=False); relevancy(item) =
         the value of the user's first test row with that item if the item is in C, else 0;
      4. a user the model was not trained on is skipped (model.recommend raises AssertionError);
      5. recommendations = [item for _, item in model.recommend(user, n=max(k), novelty=novelty,
         interaction_threshold=ignore_low_predictions_threshold)];
      6. every metric gets the arguments its __call__ names: recommendations, relevant_recommendations (the sampled
         positives), relevant_recommendation (the positive of lowest relevancy), relevancies (the relevancy of every
         item of C and of the recommendations) and k; a metric that raises (no positives, an empty list, an ideal DCG
         of 0) skips that (metric, k) for the user;
      7. each result is round(sum / count, 4), or 0 when no user counted.
    Default metrics: Precision, Recall, HitRatio and NDCG.  ds_test None (or the model's own dataset) evaluates on the
    training set.  max_concurrent_threads and verbose are accepted for compatibility and not used.

    Models with a full-catalog top-k on the device (CDAE, DMF) with integer raw item ids, the built-in metrics (strong
    relevancy) and max(k) <= 2048 are evaluated `chunk` users at a time (keyword, default 8192): topk_batch, then
    drb_eval_topk_metrics on the device computes each user's DCG, ideal DCG and hit counts; only those come back to the
    host.  The result is the same dict as the per-user loop.  Anything else runs the per-user loop over
    model.recommend, as do record= (a list that receives (user, C, recommendations) per evaluated user) and
    force_python=True.  timings= (a dict) receives, from the device path, the wall time of its host, upload and copy
    parts, the CUDA-event time of the top-k and of the metric kernel, and the per-user arrays with the evaluated users.
    """
    assert n_test_users is None or n_test_users > 0, f'The number of test users ({n_test_users}) should be > 0.'
    assert n_pos_interactions is None or n_pos_interactions > 0, \
        f'The number of positive interactions ({n_pos_interactions}) should be None or an integer > 0.'
    interaction_threshold = kwds.get('interaction_threshold', model.interaction_threshold)
    if type(k) is not list: k = [k]
    for k_ in k: assert k_ > 0, f'k ({k_}) should be > 0.'

    train_evaluation = False
    if ds_test is None or ds_test is model.interaction_dataset or ds_test is getattr(model, '_data', None):
        train_evaluation = True
        ds_test = model.interaction_dataset
    if metrics is None:
        metrics = [Precision(), Recall(), HitRatio(), NDCG()]
    assert isinstance(metrics, list), f'Expected "metrics" argument to be a list and found {type(metrics)}. ' \
        f'Should contain instances of RankingMetricABC.'
    for m in metrics:
        assert hasattr(m, 'name') and callable(m), f'Expected metric {m} to be an instance of type RankingMetricABC.'

    data = InteractionData.from_dataset(ds_test)
    users, t_indptr, t_order = _group_by_user(data)
    n_eval = len(users) if n_test_users is None else min(n_test_users, len(users))
    users, t_indptr = users[:n_eval], np.ascontiguousarray(t_indptr[:n_eval + 1])
    record = kwds.get('record', None)
    n_top = max(k)

    native_ids = np.issubdtype(data.item.dtype, np.integer)
    fast = (native_ids and hasattr(model, 'topk_batch') and hasattr(model, '_topk_device_scores') and record is None
            and not kwds.get('force_python', False) and n_top <= _TOPK_MAX
            and all(type(m) in (HitRatio, NDCG, Precision, Recall) and getattr(m, 'strong_relevancy', True)
                    for m in metrics))
    if fast:
        res = _fast_recommendation_evaluation(model, data, users, t_indptr, t_order, interaction_threshold,
                                              n_pos_interactions, train_evaluation, seed, novelty,
                                              ignore_low_predictions_threshold, metrics, k, int(kwds.get('chunk', 8192)),
                                              kwds.get('timings'))
        if res is not None:
            return res

    # ---- the per-user protocol (steps 1-3 through the same candidate generation as ranking_evaluation)
    evaluated = []           # (index, C, sampled positives, test items, test values)
    if native_ids:
        cand_off, cand, pos_off, pos, skipped, t_item, t_val = generate_candidates(
            model, data, users, t_indptr, t_order, interaction_threshold, n_pos_interactions, None, False,
            train_evaluation, seed)
        for u in np.flatnonzero(skipped == 0).tolist():
            evaluated.append((u, cand[cand_off[u]:cand_off[u + 1]].tolist(), pos[pos_off[u]:pos_off[u + 1]].tolist(),
                              t_item[t_indptr[u]:t_indptr[u + 1]].tolist(), t_val[t_indptr[u]:t_indptr[u + 1]].tolist()))
    else:
        for idx in range(n_eval):
            sl = t_order[t_indptr[idx]:t_indptr[idx + 1]]
            r_items, r_vals = data.item[sl].tolist(), data.interaction[sl].tolist()
            tpos = [it for it, v in zip(r_items, r_vals) if v >= interaction_threshold]
            res = _candidates_python(random.Random(seed + idx), list(zip(r_items, r_vals)), [], tpos, model.n_items,
                                     interaction_threshold, n_pos_interactions, None, False, train_evaluation)
            if res is not None:
                evaluated.append((idx, res[0], res[1], r_items, r_vals))

    metric_sums = {(m.name, k_): [0, 0] for m in metrics for k_ in k}
    for u, all_items, positives, r_items, r_vals in evaluated:
        user = users[u].item() if hasattr(users[u], 'item') else users[u]
        try:
            recs = model.recommend(user, n=n_top, novelty=novelty,
                                   interaction_threshold=ignore_low_predictions_threshold)
        except AssertionError:
            continue                                        # user unknown to the model
        recommendations = [item for _, item in recs]
        first_val = {}
        for it, v in zip(r_items, r_vals):
            first_val.setdefault(it, v)
        relevancies = {item: 0 for item in recommendations}
        relevancies.update({item: (first_val.get(item) or 0) for item in all_items})
        best_item = None if len(positives) == 0 else min(positives, key=lambda it: relevancies[it])
        if record is not None:
            record.append((user, list(all_items), recommendations))
        _call_metrics(metric_sums, metrics, k, recommendations, positives, best_item, relevancies)
    return _metric_results(metric_sums)


# ------------------------------------------------------------------------------------------ predictive_evaluation
class PredictiveMetricABC:
    @property
    def name(self):
        return self.__class__.__name__


class MSE(PredictiveMetricABC):
    """Mean squared error, in float64 (sklearn.metrics.mean_squared_error for one output)."""

    def __call__(self, y_true, y_pred):
        d = np.asarray(y_true, np.float64) - np.asarray(y_pred, np.float64)
        return float(np.mean(d ** 2))


class RMSE(PredictiveMetricABC):
    """Square root of MSE."""

    def __call__(self, y_true, y_pred):
        return float(np.sqrt(MSE()(y_true, y_pred)))


class MAE(PredictiveMetricABC):
    """Mean absolute error, in float64 (sklearn.metrics.mean_absolute_error for one output)."""

    def __call__(self, y_true, y_pred):
        return float(np.mean(np.abs(np.asarray(y_true, np.float64) - np.asarray(y_pred, np.float64))))


_PAIR_KERNELS = ('k_cdae_pair_scores', 'k_dmf_pair_head')


def _fast_predictive_evaluation(model, data, count_none_predictions, n_test_predictions, skip_errors, chunk, timings):
    """The rows, predictions and selection of the per-row loop in predictive_evaluation, with one predict_batch call
    over the rows that loop would predict.  Returns (y_true, y_pred) as float64 arrays."""
    t0 = time.perf_counter()
    uids, iids = model._pair_ids(data.user, data.item)
    none = (uids < 0) | (iids < 0)                         # predict() returns None (skip_errors) or raises
    if not skip_errors and none.any():
        first = int(np.argmax(none))
        if n_test_predictions is None or first < n_test_predictions:     # the loop gets there before its cap
            model.predict(data.user[first], data.item[first], skip_errors=False)   # raises predict()'s AssertionError
    rows = np.arange(len(data)) if count_none_predictions else np.flatnonzero(~none)
    if n_test_predictions is not None:
        rows = rows[:n_test_predictions]
    known = rows[~none[rows]]
    t1 = time.perf_counter()
    prof = timings is not None and getattr(model, '_ctx', None) is not None
    if prof:
        _lib.profile_read(model._ctx)                       # drop older records
        _lib.check(_lib.load().drb_ctx_profile_enable(model._ctx, 1))
    try:
        pred = model.predict_batch(data.user[known], data.item[known], skip_errors=True, chunk=chunk)
    finally:
        if prof:
            kernels = _lib.profile_read(model._ctx)
            _lib.check(_lib.load().drb_ctx_profile_enable(model._ctx, 0))
    t2 = time.perf_counter()
    y_pred = np.zeros(len(rows), np.float64)
    y_pred[~none[rows]] = pred
    y_true = np.asarray(data.interaction[rows], np.float64)
    if timings is not None:
        timings.update(host_select_s=t1 - t0, predict_batch_s=t2 - t1, n_rows=len(rows), n_predicted=len(known))
        if prof:
            timings.update(kernels_ms=kernels,
                           pair_kernel_ms=sum(v[0] for k, v in kernels.items() if k in _PAIR_KERNELS),
                           user_side_kernel_ms=sum(v[0] for k, v in kernels.items() if k not in _PAIR_KERNELS))
    return y_true, y_pred


def predictive_evaluation(model, ds_test=None, count_none_predictions=False, n_test_predictions=None, skip_errors=True,
                          metrics=None, verbose=True, **kwds):
    """Regression metrics of model.predict over the rows of ds_test (DRecPy's predictive_evaluation protocol, same
    signature).  Returns {metric.name: value}.

    The protocol:
      1. ds_test None evaluates on the model's training data (model.interaction_dataset);
      2. the rows of ds_test are taken in row order; row (user, item, value) gets
         prediction = model.predict(user, item, skip_errors=skip_errors), so with skip_errors=False an unknown user or
         item raises predict()'s AssertionError;
      3. a prediction of None (an unknown user or item, with skip_errors) is skipped, or counted as a prediction of 0
         when count_none_predictions;
      4. y_true collects the values and y_pred the predictions of the counted rows; after n_test_predictions counted
         rows (when given) no further row is predicted;
      5. every metric is computed on y_true / y_pred as float64 NumPy arrays: MSE = np.mean((y_true - y_pred) ** 2),
         RMSE = its np.sqrt, MAE = np.mean(np.abs(y_true - y_pred)) (sklearn's operations for one output);
      6. the result is {m.name: round(m(y_true, y_pred), 4)} in the order of metrics.
    Default metrics: RMSE and MSE.  verbose is accepted for compatibility and not used.

    Models with predict_batch (CDAE, DMF) make one predict_batch call over the rows step 4 counts (`chunk` pairs per
    device call, keyword) and return the same dict as the per-row loop, from the same y_pred bit for bit.  force_python=
    True runs the per-row loop.  timings= (a dict) receives y_true and y_pred from either path and, from the batched
    path, the wall time of its host selection and of predict_batch, and the CUDA-event time of every kernel launched
    (kernels_ms: {name: (ms, launches)}), summed into pair_kernel_ms (the pair kernels) and user_side_kernel_ms (the
    hidden layer / towers and the argument check).
    """
    assert n_test_predictions is None or n_test_predictions > 0, \
        f'The number of test predictions ({n_test_predictions}) should be > 0.'
    if metrics is None:
        metrics = [RMSE(), MSE()]
    assert isinstance(metrics, list), f'Expected "metrics" argument to be a list and found {type(metrics)}. ' \
        f'Should contain instances of PredictiveMetricABC.'
    for m in metrics:
        assert hasattr(m, 'name') and callable(m), f'Expected metric {m} to be an instance of type PredictiveMetricABC.'
    if ds_test is None:
        ds_test = model.interaction_dataset
    data = InteractionData.from_dataset(ds_test)
    timings = kwds.get('timings')

    if hasattr(model, 'predict_batch') and hasattr(model, '_pair_ids') and not kwds.get('force_python', False):
        y_true, y_pred = _fast_predictive_evaluation(model, data, count_none_predictions, n_test_predictions,
                                                     skip_errors, int(kwds.get('chunk', 1 << 22)), timings)
    else:
        t_list, p_list = [], []
        for user, item, value in zip(data.user.tolist(), data.item.tolist(), data.interaction.tolist()):
            prediction = model.predict(user, item, skip_errors=skip_errors)
            if prediction is None:
                if not count_none_predictions:
                    continue
                prediction = 0
            t_list.append(value)
            p_list.append(prediction)
            if n_test_predictions is not None and len(p_list) >= n_test_predictions:
                break
        y_true, y_pred = np.asarray(t_list, np.float64), np.asarray(p_list, np.float64)
    if timings is not None:
        timings.update(y_true=y_true, y_pred=y_pred)
    return {m.name: round(m(y_true, y_pred), 4) for m in metrics}
